"""The individually exposed steps -- the functions a user calls to rebuild the reference's own pipeline piece by piece
(PF:1394-1475 builds ``cape_cin`` this way) -- and the level and layer primitives, on the real-world column regimes of
tests/regime_columns.py, in float32 and float64, on every layout and through the C ABI's level strides.

Every step kernel loads its inputs as ``T``, computes in double and rounds once on store, so each is compared with
``oracle/parcel.py`` run in float64 on the SAME dtype-rounded inputs the kernel received.  The float32 and float64
calls read identical values (the regimes are float32), so one oracle serves both dtypes.

Bounds (written next to each assertion below):

* exact moves -- insert_level, shift_out_nans and its level_shift, get_layer(interpolate=False), bound_pressure, the
  NaN pattern of every output, the trap_around_zeros mask: bit for bit in both dtypes.
* computed values: ``|got - ora| <= U |ora| + REL * scale`` in float32 (U = 2^-24 is the relative error of the one
  rounding on store) and ``REL * scale`` in float64.  REL is the float64 noise of the computation: 1e-12 for the closed
  forms (a few dozen correctly rounded operations, log / exp / pow to within a few ulp: well under 1e-13 relative)
  and 1e-11 for what goes through the converged LCL iteration (the oracle's and the kernel's iterations stop at
  different, equally converged iterates).  ``scale`` is |ora| for a closed form; for a sum (trapz, cape_cin_base) it
  is the sum of the absolute terms, for an interpolated value the magnitude of the values it is interpolated between,
  since cancellation can make the result itself arbitrarily small.
* decision-boundary columns: where the oracle's decision (the LCL's side of a level, the nearest table node of a
  parcel, a crossing's side of the LCL / LFC / EL) sits within float64 noise of flipping, kernel and oracle may
  legitimately differ by a whole branch.  Those columns are found from the oracle's margin, counted and capped
  (MAX_BOUNDARY_FRACTION); they are never covered by a looser tolerance.
"""

import ctypes

import numpy as np
import pytest
import torch

import xr_double as xd
from oracle import parcel as op
from oracle import tables as otab
from oracle import thermo as th
from test_gpu_regimes_dcape_effective import AXIS_CASES, CASES, N_COLUMNS, _columns
from xarray_parcel_b200 import _lib
from xarray_parcel_b200 import parcel_functions as pf

pytestmark = pytest.mark.gpu

DTYPES = [np.float32, np.float64]
DTYPE_IDS = ["f32", "f64"]
ALL = CASES + AXIS_CASES
ALL_IDS = [c[0] for c in ALL]

# ---- bounds ----------------------------------------------------------------------------------------------------------
U = 2.0 ** -24                 # float32 unit roundoff: |round(x) - x| <= U |x|
REL = 1e-12                    # float64 noise of the closed forms and sums (relative to their scale)
REL_LCL = 1e-11                # float64 noise of what the converged LCL iteration computes
MAX_BOUNDARY_FRACTION = 0.01   # decision-boundary columns per case and output: counted, at most 1 %
PRES_STEP, TEMP_STEP = 0.5, 0.02   # the moist-adiabat table's grid (PF:447-451): nearest-node ties at half steps


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


def _np(x):
    if isinstance(x, torch.Tensor):
        x = x.cpu().numpy()
    return np.asarray(x, dtype=np.float64)


def _bits(x):
    x = x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return x.view(np.uint32 if x.dtype == np.float32 else np.uint64)


def check(got, want, f32, rel=REL, scale=None, excuse=None, what="", roundings=1):
    """NaN patterns equal and |got - want| <= (roundings U |want| if f32) + rel * scale elementwise; ``roundings``:
    float32 roundings along the chain of kernels that computed ``got`` (1 for one kernel); ``excuse``: a per-column
    mask of decision-boundary columns left out of both checks.  Returns the worst err / bound."""
    got, want = _np(got), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    keep = np.ones(want.shape, bool) if excuse is None else np.broadcast_to(~excuse, want.shape)
    gn, wn = np.isnan(got), np.isnan(want)
    bad = np.flatnonzero((gn != wn) & keep)
    assert bad.size == 0, f"{what}: NaN pattern differs at {bad.size} elements, e.g. flat {bad[:4]}: " \
                          f"got {got.flat[bad[:4]]} want {want.flat[bad[:4]]}"
    s = np.abs(want) if scale is None else np.broadcast_to(scale, want.shape)
    with np.errstate(invalid="ignore"):
        bound = (roundings * U * np.abs(want) if f32 else 0.0) + rel * s
        err = np.abs(got - want)
        over = np.flatnonzero(keep & ~wn & ~(err <= bound))
        ratio = np.where(keep & ~wn & (bound > 0), err / np.where(bound > 0, bound, 1.0), 0.0)
    assert over.size == 0, (f"{what}: {over.size} elements outside the bound, e.g. "
                            f"{[(int(i), got.flat[i], want.flat[i], bound.flat[i]) for i in over[:4]]}")
    return float(ratio.max(initial=0.0))


def check_exact(got, want, dtype, what=""):
    """Bit for bit: the oracle of an exact move is a float64 copy of dtype values, so it casts back exactly."""
    w = np.asarray(want, dtype=np.float64).astype(dtype)
    g = got.cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    assert g.dtype == dtype, (what, g.dtype)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    assert np.array_equal(_bits(g), _bits(w)) or np.array_equal(np.nan_to_num(g, nan=-7e7), np.nan_to_num(w, nan=-7e7)), \
        f"{what}: not bit-identical at {np.flatnonzero(~((g == w) | (np.isnan(g) & np.isnan(w))))[:6]}"


def cap(excuse, what):
    frac = float(np.mean(excuse)) if excuse.size else 0.0
    assert frac <= MAX_BOUNDARY_FRACTION, f"{what}: {frac:.4f} of the columns at a decision boundary"
    return int(np.sum(excuse))


def near_half_step(x, step, rel):
    """|x - nearest half-step tie of the table grid| <= rel |x|: the parcel's nearest table node is a coin toss."""
    with np.errstate(invalid="ignore"):
        r = np.abs(np.mod(x, step) - step / 2)
        return r <= rel * np.abs(x)


# ---- the cases ---------------------------------------------------------------------------------------------------------
# explicit parcels: the SB parcel of the case with these edges injected into every 41st column (from column j); the
# masked and the entirely-NaN columns of the regimes add NaN parcels of their own
EDGES = [("p", 1000.5),      # on a 0.5 hPa table node
         ("p", 1100.0),      # the table's first node
         ("p", 1120.0),      # above 1100 hPa: the adiabat lookup leaves the table
         ("p", 2.5),         # the table's last node
         ("p", 2.0),         # below it
         ("t", 173.0),       # the table's lowest temperature (dewpoint below it)
         ("t", 316.5),       # above the highest, 315.98 K
         ("td=t", None),     # saturated: the LCL is the parcel itself
         ("p", np.nan), ("t", np.nan), ("td", np.nan)]
EDGE_EVERY = 41


def _explicit(sb):
    pp, pt, pd = [x.copy() for x in sb]
    for j, (f, v) in enumerate(EDGES):
        c = slice(j, pp.size, EDGE_EVERY)
        if f == "p":
            pp[c] = v
        elif f == "t":
            pt[c] = v
            pd[c] = np.minimum(pd[c], v - 1.0)
        elif f == "td":
            pd[c] = v
        else:
            pd[c] = pt[c]
    return pp, pt, pd


class Case:
    """float32 inputs of a case, their float64 values and the parcels (float32 values), computed once."""

    def __init__(self, case_id, tables):
        i = ALL_IDS.index(case_id)
        _, regime, kw = ALL[i]
        self.id = case_id
        self.p, self.t, self.td = _columns(regime, kw, N_COLUMNS if i < len(CASES) else N_COLUMNS // 2, seed=700 + i)
        L, n = self.t.shape
        self.L, self.n = L, n
        self.shared = self.p.ndim == 1
        self.P = np.ascontiguousarray(np.broadcast_to(self.p.astype(np.float64).reshape(L, -1), (L, n)))
        self.T, self.D = self.t.astype(np.float64), self.td.astype(np.float64)
        self.compat = "1.4.1" if i % 2 == 0 else "1.6.2"
        self.opts = op.Options(op.MoistLapseLUT(tables), metpy_compat=self.compat, lcl_mode="converged")
        dat = {"pressure": self.P, "temperature": self.T, "dewpoint": self.D}
        f32 = lambda d: tuple(np.asarray(d[k], np.float32) for k in ("pressure", "temperature", "dewpoint"))  # noqa
        sb = (self.p.reshape(L, -1)[0].repeat(n // self.p.reshape(L, -1).shape[1]).astype(np.float32), self.t[0].copy(),
              self.td[0].copy())
        self.parcels = {"sb": sb, "ml": f32(op.mixed_parcel(self.P, self.T, self.D)),
                        "mu": f32(op.most_unstable_parcel(dat)), "ex": _explicit(sb)}
        self.cache = {}

    def get(self, key, fn):
        if key not in self.cache:
            self.cache[key] = fn()
        return self.cache[key]


_CASES = {}


@pytest.fixture(scope="module")
def cases(gpu_tables):
    def get(case_id):
        if case_id not in _CASES:
            _CASES[case_id] = Case(case_id, gpu_tables)
        return _CASES[case_id]
    yield get
    _CASES.clear()


def _lcl_boundary(P, lcl_p, rel):
    """Columns with a level within ``rel`` of the LCL pressure but not on it: the side of the LCL a level lies on
    (parcel_profile's p >= lcl_p, the LCL insert of PF:955) is a coin toss there."""
    with np.errstate(invalid="ignore"):
        d = np.abs(P - lcl_p[None, :])
        return ((d > 0) & (d <= rel * P)).any(axis=0)


def _lookup_boundary(lp, lt, rel):
    """Columns whose LCL sits within ``rel`` of a nearest-node tie of the table (PF:554-557)."""
    return near_half_step(lp, PRES_STEP, rel) | near_half_step(lt - 173.0, TEMP_STEP, rel)


# ---- A: pointwise steps --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_pointwise_steps_against_oracle(cases, case, dtype):
    c = cases(case)
    f32 = dtype == np.float32
    for kind, parcel in c.parcels.items():
        pp, pt, pd = [x.astype(dtype) for x in parcel]
        got = pf.lcl(pp, pt, pd, metpy_compat=c.compat)
        ora = op.lcl(*[x.astype(np.float64) for x in parcel], c.opts)
        for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature"):
            assert got[k].dtype == dtype, (k, got[k].dtype)                  # float32 in, float32 out
            check(got[k], ora[k], f32, rel=REL_LCL, what=f"lcl/{kind}/{k}")  # converged LCL: REL_LCL
        sat = ~np.isnan(ora["lcl_pressure"]) & (parcel[1] == parcel[2])
        assert np.array_equal(got["lcl_pressure"][sat], pp[sat])            # saturated: the parcel pressure itself
    # dry_lapse from level 0, on the columns' levels: one pow, REL
    P, T, D = [x.astype(dtype) for x in (c.P, c.T, c.D)]
    pt, pp = c.parcels["ex"][1].astype(dtype), c.parcels["ex"][0].astype(dtype)
    got = pf.dry_lapse(P, pt[None, :], pp[None, :])
    assert got.dtype == dtype
    check(got, th.dry_lapse(c.P, pt.astype(np.float64)[None, :], pp.astype(np.float64)[None, :]), f32,
          what="dry_lapse")
    for compat in ("1.4.1", "1.6.2"):
        got = pf.mixing_ratio(T, D, P, metpy_compat=compat)
        assert got.dtype == dtype
        ora = th.mixing_ratio_from_t_td(c.T, c.D, c.P, compat)
        check(got, ora, f32, what=f"mixing_ratio/{compat}")                 # closed form: REL
        w = ora.astype(dtype)
        got = pf.virtual_temperature(T, w)
        assert got.dtype == dtype
        check(got, th.virtual_temperature(c.T, w.astype(np.float64)), f32, what="virtual_temperature")


# ---- A: lifting ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_moist_lapse_and_parcel_profile_against_oracle(cases, case, dtype):
    """On the columns' own levels (a shared axis stays 1-D: many parcels on one axis), SB / mixed / MU / explicit."""
    c = cases(case)
    f32 = dtype == np.float32
    p = c.p.astype(dtype)
    stats = []
    for kind, parcel in c.parcels.items():
        pp, pt, pd = [x.astype(dtype) for x in parcel]
        PP, PT, PD = [x.astype(np.float64) for x in parcel]
        # moist_lapse: interpolation on the float32 table curves in double, REL; a parcel on a nearest-node tie excused
        got = pf.moist_lapse(p, pt, pp)
        assert got.dtype == dtype and got.shape == (c.L, c.n)
        tie = near_half_step(PP, PRES_STEP, REL) | near_half_step(PT - 173.0, TEMP_STEP, REL)
        check(got, c.opts.moist_lapse(c.P, PT, PP), f32, excuse=tie, what=f"moist_lapse/{kind}")
        # parcel_profile: LCL outputs REL_LCL; profiles closed forms of exact inputs (REL) except the LCL's side of a
        # level and the adiabat chosen at the LCL, both decided on a computed LCL
        r = pf.parcel_profile(p, pp, pt, pd, metpy_compat=c.compat)
        ora = op.parcel_profile(c.P, PP, PT, PD, c.opts)
        ex = _lcl_boundary(c.P, ora["lcl_pressure"], REL_LCL) | \
            _lookup_boundary(ora["lcl_pressure"], ora["lcl_temperature"], REL_LCL)
        n_ex = cap(ex, f"parcel_profile/{kind}")
        for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature"):
            assert r[k].dtype == dtype
            check(r[k], ora[k], f32, rel=REL_LCL, what=f"parcel_profile/{kind}/{k}")
        for k in ("temperature", "virtual_temperature"):
            assert r[k].dtype == dtype and r[k].shape == (c.L, c.n)
            check(r[k], ora[k], f32, excuse=ex, what=f"parcel_profile/{kind}/{k}")
        check_exact(r["pressure"], c.P, dtype, "parcel_profile/pressure")
        stats.append(f"{kind}:boundary={n_ex}")
    print(f"REGIME_STAT steps lifting {case} {np.dtype(dtype).name} " + " ".join(stats))


# ---- A + B: profile, LFC/EL, CAPE/CIN, and the reference's cape_cin rebuilt from them ------------------------------------

def _lfc_el_boundary(P, a, b, lcl_p):
    """Columns with a crossing of parcel and environment within REL of the LCL pressure: its side of the LCL
    (PF:1127, PF:1152) is a coin toss there."""
    x = op.find_intersections(P, a, b, log_x=True)["all_intersect_x"]
    with np.errstate(invalid="ignore"):
        return (np.abs(x - lcl_p[None, :]) <= REL * lcl_p[None, :]).any(axis=0)


def _cape_scale(P, env, parcel):
    """RD x the sum of the absolute trapezoids of cape_cin_base: the scale of its float64 noise (the triangles next to
    a zero are parts of these trapezoids)."""
    d = parcel - env
    with np.errstate(invalid="ignore"):
        terms = np.abs(np.diff(np.log(P), axis=0)) * (np.abs(d[:-1]) + np.abs(d[1:])) / 2
    return th.RD * np.nansum(terms, axis=0)


def _cape_boundary(P, env, parcel, lfc, el):
    """Columns where a half-area's mid pressure (PF:1347) sits within REL of the LFC or EL it is compared with."""
    areas, _ = op.trap_around_zeros(P, parcel - env, log_x=True)
    with np.errstate(invalid="ignore"):
        ax = np.exp(areas["x"])
        near = lambda v: (np.abs(ax - v[None, :]) <= REL * np.abs(v[None, :])).any(axis=0)   # noqa: E731
        return near(lfc) | near(el)


def _shifted(c, dtype):
    """(p [L, N], T, Td) of the case, shifted down to the first valid temperature on era5_masked (PF:1699-1720)."""
    P, T, D = [x.astype(dtype) for x in (c.P, c.T, c.D)]
    if "masked" not in c.id:
        return P, T, D
    r = pf.shift_out_nans({"pressure": P, "temperature": T, "dewpoint": D}, "temperature")
    ora = op.shift_out_nans({"pressure": c.P, "temperature": c.T, "dewpoint": c.D}, "temperature")
    for k in ("pressure", "temperature", "dewpoint"):
        check_exact(r[k], ora[k], dtype, f"shift_out_nans/{k}")                          # exact move
    return r["pressure"], r["temperature"], r["dewpoint"]


def _parcel(c, kind, P, T, D, dtype):
    """The parcel the reference would lift, from the library's own steps on (P, T, D)."""
    if kind == "sb":
        return P[0], T[0], D[0]
    if kind == "ml":
        m = pf.mixed_parcel(P, T, D)
        return m["pressure"], m["temperature"], m["dewpoint"]
    m = pf.most_unstable_parcel({"pressure": P, "temperature": T, "dewpoint": D})
    return m["pressure"], m["temperature"], m["dewpoint"]


def _raises(fn):
    try:
        return fn(), None
    except AssertionError as e:
        return None, str(e)


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_cape_cin_rebuilt_from_the_steps(cases, case, dtype):
    """PF:1394-1475 composed: parcel_profile_with_lcl -> lfc_el on the virtual temperatures -> cape_cin_base, for the
    SB, mixed and MU parcels; each stage against the oracle on the output of the stage before it; in float64 the
    composition equals the fused explicit-parcel cape_cin and op.cape_cin."""
    c = cases(case)
    f32 = dtype == np.float32
    P, T, D = _shifted(c, dtype)
    P64, T64, D64 = _np(P), _np(T), _np(D)
    opts = c.opts
    stats = []
    for kind in ("sb", "ml", "mu"):
        pp, pt, pd = _parcel(c, kind, P, T, D, dtype)
        PP, PT, PD = _np(pp), _np(pt), _np(pd)
        fused, fused_err = _raises(lambda: pf.cape_cin(P, T, D, pt, pp, pd, metpy_compat=c.compat))
        prof = pf.parcel_profile_with_lcl(P, T, D, pp, pt, pd, metpy_compat=c.compat)
        ora = op.parcel_profile_with_lcl(P64, T64, D64, PP, PT, PD, opts)
        ex = _lcl_boundary(P64, ora["lcl_pressure"], REL_LCL) | \
            _lookup_boundary(ora["lcl_pressure"], ora["lcl_temperature"], REL_LCL)
        for k in ("lcl_pressure", "lcl_temperature", "lcl_virtual_temperature"):
            check(prof[k], ora[k], f32, rel=REL_LCL, what=f"{kind}/{k}")
        for k in ("pressure", "temperature", "virtual_temperature", "environment_temperature",
                  "environment_dewpoint", "environment_virtual_temperature"):
            assert prof[k].dtype == dtype and prof[k].shape == (c.L + 1, c.n), k
            # the inserted LCL pressure is computed (REL_LCL), the rest closed forms and log interpolation between
            # two environment values of the same sign: REL of their magnitude, <= 2 |result| for temperatures
            check(prof[k], ora[k], f32, rel=REL_LCL if k == "pressure" else 2 * REL, excuse=ex, what=f"{kind}/{k}")
        # stage 2 on the library's stage-1 output
        Pp, Tvp, Tve = _np(prof["pressure"]), _np(prof["virtual_temperature"]), _np(prof["environment_virtual_temperature"])
        lp, ltv = _np(prof["lcl_pressure"]), _np(prof["lcl_virtual_temperature"])
        le, le_err = _raises(lambda: pf.lfc_el(prof["pressure"], prof["virtual_temperature"],
                                               prof["environment_virtual_temperature"], prof["lcl_pressure"],
                                               prof["lcl_virtual_temperature"]))
        try:
            ole, ole_err = op.lfc_el(Pp, Tvp, Tve, lp, ltv), None
        except op.ReferenceAssertion as e:
            ole, ole_err = None, str(e)
        assert le_err == ole_err, (kind, le_err, ole_err)                     # the same assertion, only there
        assert fused_err == le_err, (kind, fused_err, le_err)
        if le_err is not None:
            stats.append(f"{kind}:raises={le_err!r}")
            continue
        ex2 = _lfc_el_boundary(Pp, Tvp, Tve, lp)
        for k in ("lfc_pressure", "el_pressure", "lfc_temperature", "el_temperature"):
            assert le[k].dtype == dtype
            # crossings: (dy1 x0 - dy0 x1) / (dy1 - dy0) in ln p then exp, REL of |ln p| for the pressure (<= 8 at
            # 0.01 hPa .. 1150 hPa); the temperature interpolated between two of the same sign, REL of 2 |result|
            check(le[k], ole[k], f32, rel=8 * REL if "pressure" in k else 2 * REL, excuse=ex2,
                  what=f"{kind}/lfc_el/{k}")
        # stage 3 on the library's stage-2 output
        lfc, el = _np(le["lfc_pressure"]), _np(le["el_pressure"])
        cc = pf.cape_cin_base(prof["pressure"], prof["environment_virtual_temperature"], le["lfc_pressure"],
                              le["el_pressure"], prof["virtual_temperature"])
        occ = op.cape_cin_base(Pp, Tve, lfc, el, Tvp)
        ex3 = _cape_boundary(Pp, Tve, Tvp, lfc, el)
        scale = _cape_scale(Pp, Tve, Tvp)
        for k in ("cape", "cin"):
            assert cc[k].dtype == dtype
            check(cc[k], occ[k], f32, scale=scale, excuse=ex3, what=f"{kind}/cape_cin_base/{k}")   # a sum: REL x terms
        n_ex = cap(ex | ex2 | ex3, f"{case}/{kind}")
        if not f32:
            # float64: the composition is the fused explicit-parcel kernel's computation; 1e-9 of the terms' scale
            fcc, fprof = fused
            ref_cc, ref_prof = op.cape_cin(P64, T64, D64, PT, PP, PD, opts)
            for k in ("cape", "cin"):
                check(cc[k], fcc[k], False, rel=1e-9, scale=scale + 1.0, excuse=ex | ex2 | ex3, what=f"{kind}/fused/{k}")
                check(cc[k], ref_cc[k], False, rel=1e-9, scale=scale + 1.0, excuse=ex | ex2 | ex3, what=f"{kind}/op/{k}")
            for k in ("lfc_pressure", "el_pressure"):
                check(le[k], fprof[k], False, rel=1e-9, excuse=ex | ex2 | ex3, what=f"{kind}/fused/{k}")
                check(le[k], ref_prof[k], False, rel=1e-9, excuse=ex | ex2 | ex3, what=f"{kind}/op/{k}")
        stats.append(f"{kind}:boundary={n_ex}")
    print(f"REGIME_STAT steps composed {case} {np.dtype(dtype).name} " + " ".join(stats))


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_add_lcl_to_profile_and_cape_cin_base_options(cases, case, dtype):
    """add_lcl_to_profile (log and linear) on a parcel_profile result, and cape_cin_base with arbitrary non-crossing
    LFC / EL and every pos_cape_neg_cin / post_zero_cin combination."""
    c = cases(case)
    f32 = dtype == np.float32
    P, T, D = [x.astype(dtype) for x in (c.P, c.T, c.D)]
    pp, pt, pd = [x.astype(dtype) for x in c.parcels["ex"]]
    r = pf.parcel_profile(P, pp, pt, pd, metpy_compat=c.compat)
    w = th.mixing_ratio_from_t_td(c.T, c.D, c.P, c.compat)
    Tv = th.virtual_temperature(c.T, w).astype(dtype)
    env = {"pressure": P, "temperature": T, "dewpoint": D, "virtual_temperature": Tv}
    prof64 = {k: _np(r[k]) for k in ("pressure", "temperature", "virtual_temperature", "lcl_pressure",
                                      "lcl_temperature", "lcl_virtual_temperature")}
    env64 = {k: _np(v) for k, v in env.items()}
    for interp in ("log", "linear"):
        got = pf.add_lcl_to_profile(r, environment=env, interpolator=interp, metpy_compat=c.compat)
        ora = op.add_lcl_to_profile(prof64, env64, interp, c.opts)
        for k in ("pressure", "temperature", "virtual_temperature"):
            check_exact(got[k], ora[k], dtype, f"add_lcl/{interp}/{k}")        # insert_level of given values: exact
        for k in ("environment_temperature", "environment_dewpoint"):
            # interpolated between two values of one sign at the given LCL pressure: REL of 2 |result|
            check(got[k], ora[k], f32, rel=2 * REL, what=f"add_lcl/{interp}/{k}")
        # recomputed from the interpolated T and Td (PF:911-920) by three kernels, each rounding its output: the
        # interpolated T (U |T| <= U |Tv|), the mixing ratio from the rounded T and Td plus its own rounding (Tv moves
        # by 0.608 T w (U + 0.08 / K x U Td) < U |Tv| for w < 0.04), and Tv itself (U |Tv|): 3 U in float32; in
        # float64 a closed form of closed forms, REL of 4 |result|
        check(got["environment_virtual_temperature"], ora["environment_virtual_temperature"], f32, rel=4 * REL,
              roundings=3, what=f"add_lcl/{interp}/environment_virtual_temperature")
    # cape_cin_base on the columns' own levels with arbitrary LFC / EL (not crossings of these curves)
    tvp = _np(r["virtual_temperature"])
    rng = np.random.default_rng(11)
    lfc = rng.uniform(500.0, 1000.0, c.n).astype(dtype)
    el = (lfc * rng.uniform(0.2, 0.9, c.n)).astype(dtype)
    el[3::17] = np.nan                                                      # PF:1329: the top pressure
    scale = _cape_scale(c.P, env64["virtual_temperature"], tvp)
    ex = _cape_boundary(c.P, env64["virtual_temperature"], tvp, lfc.astype(np.float64), el.astype(np.float64))
    cap(ex, f"{case}/cape_cin_base arbitrary")
    for pos in (True, False):
        for post in (False, True):
            got = pf.cape_cin_base(P, Tv, lfc, el, r["virtual_temperature"], pos_cape_neg_cin=pos, post_zero_cin=post)
            ora = op.cape_cin_base(c.P, env64["virtual_temperature"], lfc, el, tvp, pos_cape_neg_cin=pos,
                                   post_zero_cin=post)
            for k in ("cape", "cin"):
                check(got[k], ora[k], f32, scale=scale, excuse=ex, what=f"cape_cin_base/{pos}/{post}/{k}")


# ---- A: level primitives -------------------------------------------------------------------------------------------------

def _with_zeros(y, every=7):
    """``y`` with exact zeros on one level of every ``every``-th column (two levels in every other such column)."""
    y = y.copy()
    L, n = y.shape
    cols = np.arange(1, n, every)
    y[(cols * 3) % (L - 1), cols] = 0.0
    y[((cols * 3) % (L - 1) + 1)[::2], cols[::2]] = 0.0
    return y


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_level_primitives_against_oracle(cases, case, dtype):
    """trapz, find_intersections, trap_around_zeros, linear / log_interp, interp1d_numba on the case's columns, with
    exact zeros at levels and crossings in the masked and extrapolated levels (they are part of the columns)."""
    c = cases(case)
    f32 = dtype == np.float32
    p = c.p.astype(dtype)                                   # shared axes stay 1-D
    y = _with_zeros((c.t - np.float32(273.15)).astype(np.float32)).astype(dtype)
    Y = y.astype(np.float64)
    T, D = c.t.astype(dtype), c.td.astype(dtype)
    b = (c.td + np.float32(4.0)).astype(dtype)
    B = b.astype(np.float64)
    lx = np.log(c.P)
    # find_intersections: ix from (dy1 x0 - dy0 x1) / (dy1 - dy0): REL of |x0| + |x1| (of |ln x0| + |ln x1| before
    # the exp with log_x, then relative); iy interpolated between a0 and a1: REL of |a0| + |a1|
    for log_x in (False, True):
        got = pf.find_intersections(p, T, b, log_x=log_x)
        ora = op.find_intersections(c.P, c.T, B, log_x=log_x)
        xs = (np.abs(lx[:-1]) + np.abs(lx[1:])) if log_x else (c.P[:-1] + c.P[1:])
        ys = np.abs(c.T[:-1]) + np.abs(c.T[1:])
        for k, v in ora.items():
            assert got[k].dtype == dtype and got[k].shape == (c.L - 1, c.n), k
            if k.endswith("_x"):
                sc = xs * np.abs(v) if log_x else xs
            else:
                sc = ys
            check(got[k], v, f32, scale=sc, what=f"find_intersections/{log_x}/{k}")
    # trap_around_zeros: mask bit for bit; x / dx / x_from / x_to in ln p, REL of |ln p0| + |ln p1| (+ |result|);
    # area = y / 2 * |dx|: REL of |y| (|ln p0| + |ln p1|)
    for log_x in (True, False):
        areas, mask = pf.trap_around_zeros(p, y, log_x=log_x)
        oa, om = op.trap_around_zeros(c.P, Y, log_x=log_x)
        assert np.array_equal(np.asarray(mask), om), f"trap_around_zeros mask log_x={log_x}"
        xx = lx if log_x else c.P
        pad = lambda a: np.concatenate([a, np.full((1, c.n), np.nan)])               # noqa: E731
        sx = np.abs(xx[:-1]) + np.abs(xx[1:])
        sx2 = np.concatenate([pad(sx), sx])                                             # before rows, after rows
        yv = np.concatenate([Y, Y[1:]])
        for k, v in oa.items():
            assert areas[k].dtype == dtype and areas[k].shape == (2 * c.L - 1, c.n), k
            sc = np.abs(yv) * sx2 if k == "area" else sx2 + np.abs(v)
            check(areas[k], v, f32, scale=sc, what=f"trap_around_zeros/{log_x}/{k}")
    # trapz along pressure of T, Td and pressure itself, sign -1 / 0 / +1, with and without the mask above
    dat = {"pressure": p, "temperature": y, "dewpoint": D}
    dat64 = {"pressure": c.P, "temperature": Y, "dewpoint": c.D}
    dp = np.abs(np.diff(c.P, axis=0))
    for m in (None, om):
        for sign in (-1, 0, 1):
            got = pf.trapz(dat, "pressure", mask=m, only_positive=sign > 0, only_negative=sign < 0)
            ora = op.trapz(dat64, "pressure", mask=m, only_positive=sign > 0, only_negative=sign < 0)
            for k, v in ora.items():
                with np.errstate(invalid="ignore"):
                    sc = np.nansum(dp * (np.abs(dat64[k][:-1]) + np.abs(dat64[k][1:])) / 2, axis=0)
                check(got[k], v, f32, scale=sc, what=f"trapz/{sign}/{m is not None}/{k}")    # a sum: REL x terms
    # linear / log interp at one pressure per column: some exactly on a level, some outside the column (NaN)
    rng = np.random.default_rng(5)
    at = rng.uniform(50.0, 1000.0, c.n).astype(dtype)
    at[::13] = p.reshape(c.L, -1)[c.L // 3][0] if c.shared else p[c.L // 3, ::13]
    at[7::29] = 1200.0
    for log in (False, True):
        fn = pf.log_interp if log else pf.linear_interp
        got = fn(T, p, at)
        ora = (op.log_interp if log else op.linear_interp)({"x": c.T}, c.P, at.astype(np.float64))["x"]
        assert got.dtype == dtype
        check(got, ora, f32, rel=2 * REL, what=f"interp/{log}")     # between two temperatures: REL of 2 |result|
    # interp1d_numba (numpy.interp along the last axis): one rounding of numpy.interp of the same values
    xp = np.sort(rng.uniform(0.0, 100.0, 40)).astype(dtype)
    fp = rng.normal(0.0, 50.0, (c.n, 40)).astype(dtype)
    a = rng.uniform(-5.0, 105.0, (c.n, 25)).astype(dtype)
    a[:, 0] = xp[3]                                                       # exact node hits
    got = pf.interp1d_numba(a, xp, fp)
    assert got.dtype == dtype
    want = np.stack([np.interp(a[i].astype(np.float64), xp.astype(np.float64), fp[i].astype(np.float64))
                     for i in range(c.n)])
    sc = np.max(np.abs(fp.astype(np.float64)), axis=1, keepdims=True) * np.ones_like(want)
    check(got, want, f32, scale=sc, what="interp1d")                 # f0 + slope (x - x0): REL of max |fp|


# ---- A: layer primitives ---------------------------------------------------------------------------------------------------

def _get_layer_at(dat, top):
    """op.get_layer(interpolate=True) at a given top (the kernel's, rounded to the dtype: it is stored as T before the
    level is inserted)."""
    bottom = op.nanmax(dat["pressure"])
    lev = op.log_interp(dat, dat["pressure"], top)
    lev["pressure"] = top
    d = op.insert_level(dat, lev, "pressure")
    with np.errstate(invalid="ignore"):
        keep = (d["pressure"] <= bottom[None, :]) & (d["pressure"] >= top[None, :])
    return {k: np.where(keep, v, np.nan) for k, v in d.items()}


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_layer_primitives_against_oracle(cases, case, dtype):
    c = cases(case)
    f32 = dtype == np.float32
    p = c.p.astype(dtype)
    P, T, D = [x.astype(dtype) for x in (c.P, c.T, c.D)]
    dat = {"pressure": p, "temperature": T, "dewpoint": D}
    dat64 = {"pressure": c.P, "temperature": c.T, "dewpoint": c.D}
    for depth in (50, 100, 300, 2000):                                    # 2000 hPa: deeper than any column
        got = pf.get_layer(dat, depth=depth, interpolate=False)
        ora = op.get_layer(dat64, depth=depth, interpolate=False)
        for k in ora:
            check_exact(got[k], ora[k], dtype, f"get_layer/False/{depth}/{k}")     # a selection: exact
        top = np.broadcast_to(pf.bound_pressure(p, depth=depth), (c.n,))    # a shared axis has one bound
        check_exact(top, op.bound_pressure(c.P, op.nanmax(c.P) - depth), dtype, f"bound_pressure/{depth}")
        got = pf.get_layer(dat, depth=depth, interpolate=True)
        top = (op.nanmax(c.P) - depth).astype(dtype).astype(np.float64)
        ora = _get_layer_at(dat64, top)
        for k in ora:
            # the inserted level interpolated between two values of one sign (REL of 2 |result|); the rest exact
            check(got[k], ora[k], f32, rel=2 * REL, what=f"get_layer/True/{depth}/{k}")
    # mixed_layer over six variables (two launches) and mixed_parcel's six outputs: sums of positive terms
    # (temperatures, pressures, mixing ratios) over the lowest 100 hPa divided by its depth, REL of |result|; the
    # dewpoint a log of that: REL
    w = th.saturation_mixing_ratio(c.P, c.D)
    theta = th.potential_temperature(c.P, c.T)
    six = {"pressure": p, "temperature": T, "dewpoint": D, "theta": theta.astype(dtype), "mixing_ratio": w.astype(dtype),
           "temperature_again": T}
    six64 = {k: _np(v) if k != "pressure" else c.P for k, v in six.items()}
    got = pf.mixed_layer(six, depth=100)
    ora = op.mixed_layer(six64, depth=100)
    for k, v in ora.items():
        assert got[k].dtype == dtype
        check(got[k], v, f32, rel=2 * REL, what=f"mixed_layer/{k}")
    assert np.array_equal(_bits(got["temperature"]), _bits(got["temperature_again"]))  # same sum in either launch
    got = pf.mixed_parcel(p, T, D, depth=100)
    ora = op.mixed_parcel(c.P, c.T, c.D, depth=100)
    for k, v in ora.items():
        assert got[k].dtype == dtype
        check(got[k], v, f32, rel=4 * REL, what=f"mixed_parcel/{k}")
    # valid_data: good, tied and reversed levels
    assert pf.valid_data({"pressure": p}) is True
    bad = P.copy()
    bad[3, 10] = bad[2, 10]
    with pytest.raises(AssertionError, match="Pressures must decrease"):
        pf.valid_data({"pressure": bad})
    with pytest.raises(AssertionError, match="Pressures must decrease"):
        pf.valid_data({"pressure": np.ascontiguousarray(p[::-1])})


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_bound_pressure_tie_takes_the_larger_pressure(dtype):
    """PF:208-227: two levels equally far from bottom - depth -> the larger pressure, also in get_layer."""
    p = np.array([[1000.0, 1000.0], [950.0, 960.0], [925.0, 925.0], [900.0, 900.0], [850.0, 850.0], [700.0, 700.0]],
                 dtype=dtype)
    top = pf.bound_pressure(p, depth=87.5)                                # 912.5: 925 and 900 tie
    assert top.tolist() == [925.0, 925.0]
    lay = pf.get_layer({"pressure": p, "temperature": p - 700}, depth=87.5, interpolate=False)
    assert np.array_equal(np.isnan(lay["pressure"][:, 0]), [False, False, False, True, True, True])


# ---- A: exact moves ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", ALL_IDS)
def test_insert_level_and_shift_out_nans_are_exact(cases, case, dtype):
    c = cases(case)
    p = c.p.astype(dtype)
    T, D = c.t.astype(dtype), c.td.astype(dtype)
    rng = np.random.default_rng(9)
    lev_p = rng.uniform(100.0, 1100.0, c.n).astype(dtype)
    P0 = c.P
    lev_p[::11] = P0[c.L // 2, ::11]                                       # on a level: the insert tie of PF:955
    lev_p[1::11] = P0[0, 1::11]                                           # on the surface level
    lev_p[2::37] = np.nan
    lev = {"pressure": lev_p, "temperature": rng.uniform(200, 300, c.n).astype(dtype),
           "dewpoint": rng.uniform(190, 290, c.n).astype(dtype)}
    got = pf.insert_level({"pressure": p, "temperature": T, "dewpoint": D}, lev, "pressure")
    ora = op.insert_level({"pressure": c.P, "temperature": c.T, "dewpoint": c.D},
                          {k: v.astype(np.float64) for k, v in lev.items()}, "pressure")
    for k in ora:
        check_exact(got[k], ora[k], dtype, f"insert_level/{k}")
    x = {"pressure": p, "temperature": T, "dewpoint": D}                  # a shared axis stays 1-D
    got = pf.shift_out_nans(x, "temperature")
    ora = op.shift_out_nans({"pressure": c.P, "temperature": c.T, "dewpoint": c.D}, "temperature")
    for k in ora:
        check_exact(got[k], ora[k], dtype, f"shift_out_nans/{k}")
    # level_shift: the number of leading NaN temperature levels (all L where the column is NaN throughout)
    ctx = _lib.get_context(0)
    t_dev = torch.from_numpy(np.ascontiguousarray(T)).cuda()
    _, shift = ctx.shift_out_nans(t_dev, [t_dev])
    lead = np.argmax(~np.isnan(c.t), axis=0)
    lead[np.isnan(c.t).all(axis=0)] = c.L
    assert np.array_equal(shift.cpu().numpy(), lead)


# ---- C: layouts ----------------------------------------------------------------------------------------------------------------

def _yx(n):
    m = n // 2
    y = max(d for d in range(1, int(m ** 0.5) + 1) if m % d == 0)
    return y, m // y


class Layout:
    """Puts level-major [L, N] fields and [N] column values into one layout and takes results back to level-major
    NumPy."""

    def __init__(self, kind, L, n, dtype):
        self.kind, self.L, self.n, self.dtype = kind, L, n, dtype
        self.vert_axis = 1 if kind in ("nl", "4d") else 0

    def prof(self, x, name=None):
        x = np.asarray(x, dtype=self.dtype)
        if x.ndim == 1 and x.shape[0] == self.L and self.kind != "xr":
            return x                                                    # a shared axis stays as it is
        if self.kind == "nl":
            return np.ascontiguousarray(x.T)
        if self.kind == "4d":
            y, xx = _yx(self.n)
            return np.ascontiguousarray(x.reshape(self.L, 2, y, xx).transpose(1, 0, 2, 3))
        if self.kind in ("cuda", "cpu"):
            t = torch.from_numpy(np.ascontiguousarray(x))
            return t.cuda() if self.kind == "cuda" else t
        if self.kind == "xr":
            if x.ndim == 1:
                return xd.DataArray(x, dims=("lev",), coords={"lev": np.arange(self.L) + 3})
            return xd.DataArray(x, dims=("lev", "col"), coords={"lev": np.arange(self.L) + 3,
                                                                 "col": np.arange(self.n)})
        return x

    def col(self, x):
        x = np.asarray(x, dtype=self.dtype)
        if self.kind == "4d":
            return x.reshape(2, *_yx(self.n))
        if self.kind in ("cuda", "cpu"):
            t = torch.from_numpy(np.ascontiguousarray(x))
            return t.cuda() if self.kind == "cuda" else t
        if self.kind == "xr":
            return xd.DataArray(x, dims=("col",), coords={"col": np.arange(self.n)})
        return x

    def back(self, r, first=3):
        """Result -> level-major NumPy; checks the array type, device, dtype and the xarray vertical labels."""
        if self.kind in ("cuda", "cpu"):
            assert isinstance(r, torch.Tensor) and r.is_cuda == (self.kind == "cuda"), type(r)
            r = r.cpu().numpy()
        elif self.kind == "xr" and not isinstance(r, np.ndarray):              # lcl hands back plain arrays
            assert isinstance(r, xd.DataArray), type(r)
            if "lev" in r.dims:
                labels = np.asarray(r["lev"].values)
                assert np.array_equal(labels, np.arange(labels.size) + first), labels[:5]
            r = np.asarray(r.data)
        else:
            assert isinstance(r, np.ndarray), type(r)
        r = np.asarray(r)
        assert r.dtype == self.dtype, r.dtype
        if self.kind == "nl":
            return r.T if r.ndim == 2 else r
        if self.kind == "4d":
            return r.transpose(1, 0, 2, 3).reshape(r.shape[1], -1) if r.ndim == 4 else r.reshape(-1)
        return r


def _calls(c, lay, p):
    """(name, thunk) of every public function of section A in layout ``lay``; ``p`` is the pressure to pass ([L, N]
    or the shared [L]).  Each thunk returns a dict of results still in the layout."""
    F = lay.prof
    S = lay.col
    va = {"vert_axis": lay.vert_axis} if lay.kind != "xr" else {"vert_dim": "lev"}
    vd = {"dim": "lev"} if lay.kind == "xr" else {"vert_axis": lay.vert_axis}
    pp, pt, pd = c.parcels["ex"]
    T, D = c.t, c.td
    y = _with_zeros(c.t - np.float32(273.15))
    ds = lambda r: dict(r.items()) if hasattr(r, "items") else {"out": r}      # noqa: E731
    lcl_p = np.asarray(op.lcl(pp.astype(np.float64), pt.astype(np.float64), pd.astype(np.float64),
                              c.opts)["lcl_pressure"], np.float32)
    prof_t = c.opts.moist_lapse(c.P, pt.astype(np.float64), pp.astype(np.float64)).astype(np.float32)
    T_env = np.where(np.isnan(prof_t), np.float32(np.nan), T)          # NaN parcels: no PF:1149 assertion
    at = np.linspace(300.0, 900.0, c.n).astype(np.float32)
    return [
        ("lcl", lambda: ds(pf.lcl(S(pp), S(pt), S(pd)))),
        ("moist_lapse", lambda: ds(pf.moist_lapse(F(p), S(pt), S(pp), **va))),
        ("parcel_profile", lambda: ds(pf.parcel_profile(F(p), S(pp), S(pt), S(pd), **va))),
        ("parcel_profile_with_lcl", lambda: ds(pf.parcel_profile_with_lcl(F(p), F(T), F(D), S(pp), S(pt), S(pd), **va))),
        ("lfc_el", lambda: ds(pf.lfc_el(F(p), F(prof_t), F(T_env), S(lcl_p), S(pt), **va))),
        ("cape_cin_base", lambda: ds(pf.cape_cin_base(F(p), F(T), S(lcl_p), S(lcl_p * 0.4), F(prof_t), **va))),
        ("insert_level", lambda: ds(pf.insert_level({"pressure": F(p), "temperature": F(T)},
                                                    {"pressure": S(lcl_p), "temperature": S(pt)}, "pressure", **va))),
        ("shift_out_nans", lambda: ds(pf.shift_out_nans({"pressure": F(p), "temperature": F(T)}, "temperature",
                                                        **vd))),
        ("trapz", lambda: ds(pf.trapz({"pressure": F(p), "temperature": F(y)}, "pressure", **vd))),
        ("find_intersections", lambda: ds(pf.find_intersections(F(p), F(T), F(D + np.float32(4.0)), log_x=True, **vd))),
        ("trap_around_zeros", lambda: ds(pf.trap_around_zeros(F(p), F(y), **vd)[0])),
        ("log_interp", lambda: ds(pf.log_interp(F(T), F(p), S(at), **vd))),
        ("get_layer", lambda: ds(pf.get_layer({"pressure": F(p), "temperature": F(T)}, depth=100, **va))),
        ("get_layer_nointerp", lambda: ds(pf.get_layer({"pressure": F(p), "temperature": F(T)}, depth=100,
                                                       interpolate=False, **va))),
        ("bound_pressure", lambda: ds(pf.bound_pressure(F(p), depth=100, **va))),
        ("mixed_layer", lambda: ds(pf.mixed_layer({"pressure": F(p), "temperature": F(T), "dewpoint": F(D)}, **va))),
        ("mixed_parcel", lambda: ds(pf.mixed_parcel(F(p), F(T), F(D), **va))),
    ]


LAYOUTS = ["nl", "4d", "cuda", "cpu", "xr", "axis1d"]
LAYOUT_CASES = ["terrain_L40", "cold_era5_masked"]


@pytest.fixture()
def xr_pf():
    xd.install()
    try:
        yield
    finally:
        xd.uninstall()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_every_step_on_every_layout_gives_the_level_major_bits(cases, case, dtype, layout, request):
    """Each public function in each layout: the same bits as the level-major NumPy call, in the input's dtype.  A
    shared 1-D pressure axis gives the same bits as the broadcast [L, N] pressure."""
    c = cases(case)
    if layout == "axis1d" and not c.shared:
        pytest.skip("per-column pressure: no shared axis to compare with")
    base_lay = Layout("lm", c.L, c.n, dtype)
    p_full = c.P.astype(np.float32)
    # the level-major reference: [L, N] pressure (the broadcast axis where the case has one)
    ref = {name: {k: base_lay.back(v) for k, v in fn().items()} for name, fn in _calls(c, base_lay, p_full)}
    if layout == "xr":
        request.getfixturevalue("xr_pf")
    lay = Layout("lm" if layout == "axis1d" else layout, c.L, c.n, dtype)
    p = c.p if layout in ("axis1d", "xr") and c.shared else p_full
    for name, fn in _calls(c, lay, p):               # (xr_double.install() reloads parcel_functions in place)
        got = fn()
        for k, want in ref[name].items():
            # find_intersections labels its L - 1 rows by the upper level of each interval (PF:1026)
            g = lay.back(got[k], first=4 if name == "find_intersections" else 3)
            if name == "bound_pressure" and g.size == 1:
                g = np.broadcast_to(g, want.shape)   # one shared axis, one bound
            assert g.shape == want.shape, (name, k, g.shape, want.shape)
            assert np.array_equal(_bits(g), _bits(want)), (name, k)


# ---- E: flags ----------------------------------------------------------------------------------------------------------------

def test_lfc_el_clears_flags_left_by_earlier_calls(ctx, cases):
    c = cases("terrain")
    dv = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).cuda()      # noqa: E731
    P, T = c.P[:, :64], c.T[:, :64].copy()
    parcel = c.opts.moist_lapse(P, T[0], P[0])
    bad = parcel.copy()
    bad[:, 9] = np.nan                       # no level with both temperatures while the environment has some: PF:1149
    with pytest.raises(op.ReferenceAssertion, match="Top temperature is NaN."):
        op.lfc_el(P, bad, T, P[0], T[0])
    ctx.take_flags()
    ctx.lfc_el(dv(P), dv(bad), dv(T), dv(P[0]), dv(T[0]))             # a direct call leaves its flag behind
    r = pf.lfc_el(P, parcel, T, P[0], T[0])                            # good input must not raise
    want = op.lfc_el(P, parcel, T, P[0], T[0])
    for k in want:
        assert np.array_equal(np.isnan(r[k]), np.isnan(want[k])), k
    with pytest.raises(AssertionError, match="Top temperature is NaN."):
        pf.lfc_el(P, bad, T, P[0], T[0])


# ---- D: the C ABI's strides -------------------------------------------------------------------------------------------------

GUARD = 7                       # guard columns on each side of the window in the input allocation
PATTERN32, PATTERN64 = 0x7FA5A5A5, 0x7FF5A5A5A5A5A5A5    # NaN payloads no kernel computes


class Wide:
    """One flat device allocation sized for [rows, max(W_in, W_out)]; ``view(rows, w)`` a [rows, w] view of it."""

    def __init__(self, rows, wmax, dtype, fill):
        self.dt = torch.float32 if dtype == np.float32 else torch.float64
        self.flat = torch.empty(rows * wmax, dtype=self.dt, device="cuda")
        if fill == "poison":
            v = torch.tensor([float("nan"), 1e30, -1e30], dtype=self.dt, device="cuda")
            self.flat.copy_(v.repeat(rows * wmax // 3 + 1)[:rows * wmax])
        else:
            it = torch.int32 if self.dt == torch.float32 else torch.int64
            pat = PATTERN32 if self.dt == torch.float32 else PATTERN64
            self.flat.view(it).fill_(pat)

    def view(self, rows, w):
        return self.flat[:rows * w].view(rows, w)


def _window_call(ctx, dtype, L, n, ins, outs, call, out_stride=True):
    """Run ``call(ptr_in, ls, ptr_out, ols)`` on a window of n columns at offset GUARD: inputs [L, n] (name -> CUDA
    tensor, or [n] for per-column values) in a poisoned [L, W] allocation, outputs (name -> rows or 0 for [n]) in a
    pattern-filled [rows, W'] allocation; every allocation sized for max(W, W').  Returns {name: [rows, n]} and checks
    that the pattern survives outside the window."""
    W = n + 2 * GUARD
    Wo = n + 3 * GUARD if out_stride else W          # an entry without an output stride writes with level_stride
    Wm, Lm = max(W, Wo), max([L] + [r for r in outs.values()] + [1]) + 1
    keep = []
    ptr_in = {}
    for k, v in ins.items():
        a = Wide(Lm, Wm, dtype, "poison")
        if v.dim() == 1:
            a.flat[GUARD:GUARD + n] = v
            ptr_in[k] = a.flat[GUARD:].data_ptr()
        else:
            a.view(v.shape[0], W)[:, GUARD:GUARD + n] = v
            ptr_in[k] = a.view(v.shape[0], W)[:, GUARD:].data_ptr()
        keep.append(a)
    bufs, ptr_out = {}, {}
    for k, rows in outs.items():
        b = Wide(Lm, Wm, dtype, "pattern")
        bufs[k] = (b, rows)
        ptr_out[k] = b.flat[GUARD:].data_ptr()
    call(ptr_in, W, ptr_out, Wo)
    torch.cuda.synchronize()
    res = {}
    for k, (b, rows) in bufs.items():
        it = torch.int32 if b.dt == torch.float32 else torch.int64
        pat = PATTERN32 if b.dt == torch.float32 else PATTERN64
        bits = b.flat.view(it).clone()
        if rows == 0:
            res[k] = b.flat[GUARD:GUARD + n].clone()
            bits[GUARD:GUARD + n] = pat
        else:
            v = bits[:rows * Wo].view(rows, Wo)
            res[k] = b.view(rows, Wo)[:, GUARD:GUARD + n].clone()
            v[:, GUARD:GUARD + n] = pat
        assert bool((bits == pat).all()), f"{k}: an element outside the window was written"
    return res


def _ptrs(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*ptrs)


def _step_entries(ctx, dtype):
    """name -> (inputs builder, outputs {name: rows}, call(ptr_in, ls, ptr_out, ols, L, n), compact reference)."""
    lib, h = ctx.lib, ctx.handle
    code = _lib._dtype_code(torch.empty(0, dtype=torch.float32 if dtype == np.float32 else torch.float64))
    opts = _lib.make_options()
    st = lambda: ctx._stream()                                                    # noqa: E731
    E = {}
    E["moist_lapse"] = (["pressure", "pt", "pp"], lambda L: {"out": L},
                        lambda pi, ls, po, ols, L, n: lib.xp_moist_lapse(h, pi["pressure"], ls, L, n, code, pi["pt"],
                                                                          pi["pp"], po["out"], ols, st()),
                        lambda d: {"out": ctx.moist_lapse(d["pressure"], d["pt"], d["pp"])})

    def pprof(pi, ls, po, ols, L, n):
        pin = _lib.XpParcelIn(pi["pp"], pi["pt"], pi["pd"])
        return lib.xp_parcel_profile(h, pi["pressure"], ls, L, n, code, ctypes.byref(pin), ctypes.byref(opts),
                                     po["t"], po["tv"], ols, po["lp"], po["lt"], po["ltv"], st())
    E["parcel_profile"] = (["pressure", "pp", "pt", "pd"], lambda L: {"t": L, "tv": L, "lp": 0, "lt": 0, "ltv": 0}, pprof,
                           lambda d: dict(zip(["t", "tv", "lp", "lt", "ltv"], [
                               ctx.parcel_profile(d["pressure"], d["pp"], d["pt"], d["pd"])[k] for k in
                               ("temperature", "virtual_temperature", "lcl_pressure", "lcl_temperature",
                                "lcl_virtual_temperature")])))
    E["lfc_el"] = (["pressure", "a", "b", "lp", "lt"], lambda L: {"lfc": 0, "lft": 0, "el": 0, "elt": 0},
                   lambda pi, ls, po, ols, L, n: lib.xp_lfc_el(h, pi["pressure"], pi["a"], pi["b"], ls, L, n, code,
                                                               pi["lp"], pi["lt"], po["lfc"], po["lft"], po["el"],
                                                               po["elt"], st()),
                   lambda d: dict(zip(["lfc", "lft", "el", "elt"], ctx.lfc_el(d["pressure"], d["a"], d["b"], d["lp"],
                                                                               d["lt"]).values())))
    E["cape_cin_base"] = (["pressure", "b", "a", "lp", "el"], lambda L: {"cape": 0, "cin": 0},
                          lambda pi, ls, po, ols, L, n: lib.xp_cape_cin_base(h, pi["pressure"], pi["b"], pi["a"], ls, L,
                                                                             n, code, pi["lp"], pi["el"],
                                                                             ctypes.byref(opts), po["cape"], po["cin"],
                                                                             st()),
                          lambda d: dict(zip(["cape", "cin"], ctx.cape_cin_base(d["pressure"], d["b"], d["lp"], d["el"],
                                                                                 d["a"]).values())))

    def fi(pi, ls, po, ols, L, n):
        o = _lib.XpIntersectionsOut(*[po[k] for k in _lib.INTERSECTION_FIELDS])
        return lib.xp_find_intersections(h, pi["pressure"], ls, 0, pi["a"], pi["b"], ls, ols, L, n, code, 1,
                                         ctypes.byref(o), st())
    E["find_intersections"] = (["pressure", "a", "b"], lambda L: {k: L - 1 for k in _lib.INTERSECTION_FIELDS}, fi,
                               lambda d: ctx.find_intersections(d["pressure"], d["a"], d["b"], log_x=True))

    masks = []

    def taz(pi, ls, po, ols, L, n):
        masks.append(torch.empty((L, n), dtype=torch.uint8, device="cuda"))    # contiguous whatever ols is
        o = _lib.XpZeroAreasOut(*([po[k] for k in _lib.ZERO_AREA_FIELDS] + [masks[-1].data_ptr()]))
        return lib.xp_trap_around_zeros(h, pi["pressure"], ls, 0, pi["y"], ls, ols, L, n, code, 1, ctypes.byref(o),
                                        st())
    E["trap_around_zeros"] = (["pressure", "y"], lambda L: {k: 2 * L - 1 for k in _lib.ZERO_AREA_FIELDS}, taz,
                              lambda d: ctx.trap_around_zeros(d["pressure"], d["y"])[0])

    def ins(pi, ls, po, ols, L, n):
        return lib.xp_insert_level(h, pi["pressure"], ls, 0, pi["lp"], _ptrs([pi["a"]]),
                                   _ptrs([pi["lt"]]), _ptrs([po["a"]]), 1, po["c"], ls, ols, L, n,
                                   code, st())
    E["insert_level"] = (["pressure", "a", "lp", "lt"], lambda L: {"c": L + 1, "a": L + 1}, ins,
                         lambda d: dict(zip(["c", "a"], (lambda r: (r[0], r[1][0]))(
                             ctx.insert_level(d["pressure"], d["lp"], [d["a"]], [d["lt"]])))))

    def tz(pi, ls, po, ols, L, n):
        return lib.xp_trapz(h, pi["pressure"], ls, 0, _ptrs([pi["a"], pi["b"]]),
                            _ptrs([po["a"], po["b"]]), 2, ls, L, n, code, None, 0, 0, st())
    E["trapz"] = (["pressure", "a", "b"], lambda L: {"a": 0, "b": 0}, tz,
                  lambda d: dict(zip(["a", "b"], ctx.trapz(d["pressure"], [d["a"], d["b"]]))))

    def ml(pi, ls, po, ols, L, n):
        return lib.xp_mixed_layer(h, pi["pressure"], ls, 0, _ptrs([pi["a"], pi["pressure"]]),
                                  _ptrs([po["a"], po["p"]]), 2, 1, ls, L, n, code, 100.0, st())
    E["mixed_layer"] = (["pressure", "a"], lambda L: {"a": 0, "p": 0}, ml,
                        lambda d: dict(zip(["a", "p"], ctx.mixed_layer(d["pressure"], [d["a"], d["pressure"]],
                                                                       pressure_field=1))))

    def il(pi, ls, po, ols, L, n):
        return lib.xp_interp_levels(h, pi["pressure"], ls, 0, _ptrs([pi["a"]]), _ptrs([po["a"]]), 1,
                                    ls, L, n, code, pi["lp"], 0.0, 1, st())
    E["interp_levels"] = (["pressure", "a", "lp"], lambda L: {"a": 0}, il,
                          lambda d: {"a": ctx.interp_levels(d["pressure"], [d["a"]], d["lp"], log=True)[0]})

    def so(pi, ls, po, ols, L, n):
        return lib.xp_shift_out_nans(h, pi["a"], _ptrs([pi["a"], pi["b"]]), _ptrs([po["a"], po["b"]]),
                                     2, ls, L, n, code, None, st())
    E["shift_out_nans"] = (["a", "b"], lambda L: {"a": L, "b": L}, so, None)
    return E


def _step_inputs(c, dtype):
    """Device inputs [L, N] / [N] of every entry, from a masked ERA5 case (NaN levels, crossings below ground)."""
    dt = torch.float32 if dtype == np.float32 else torch.float64
    dv = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dt).cuda()          # noqa: E731
    pp, pt, pd = c.parcels["sb"]
    a = c.opts.moist_lapse(c.P, pt.astype(np.float64), pp.astype(np.float64))
    lp = op.lcl(pp, pt, pd, c.opts)
    return {"pressure": dv(c.P), "pt": dv(pt), "pp": dv(pp), "pd": dv(pd), "a": dv(a), "b": dv(c.T),
            "y": dv(_with_zeros(c.t - np.float32(273.15))), "lp": dv(lp["lcl_pressure"]),
            "lt": dv(lp["lcl_temperature"]), "el": dv(np.full(c.n, 300.0))}


STEP_ENTRIES = ["moist_lapse", "parcel_profile", "lfc_el", "cape_cin_base", "find_intersections", "trap_around_zeros",
                "insert_level", "trapz", "mixed_layer", "interp_levels", "shift_out_nans"]
HAS_OUT_STRIDE = {"moist_lapse", "parcel_profile", "find_intersections", "trap_around_zeros", "insert_level"}


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("entry", STEP_ENTRIES)
def test_c_abi_column_window_equals_the_compact_call(ctx, cases, entry, dtype):
    """A window of n columns of a wider [L, W] allocation (level_stride W > n; outputs with stride W' > W where the
    entry has an output stride), columns outside poisoned, output elements outside pre-filled: the window's results are
    the compact call's bits, and no element outside the window changes."""
    c = cases("terrain_era5_masked")
    n = 300
    d = {k: (v[:, :n] if v.dim() == 2 else v[:n]).contiguous() for k, v in _step_inputs(c, dtype).items()}
    names, outs_of, call, compact = _step_entries(ctx, dtype)[entry]
    L = c.L
    ins = {k: d[k] for k in names}
    ctx.take_flags()
    res = _window_call(ctx, dtype, L, n, ins, outs_of(L), lambda pi, ls, po, ols: ctx._check(call(pi, ls, po, ols, L, n),
                                                                                              entry),
                       out_stride=entry != "shift_out_nans")
    if entry == "shift_out_nans":
        want, _ = ctx.shift_out_nans(d["a"], [d["a"], d["b"]])
        want = {"a": want[0], "b": want[1]}
    else:
        want = compact(d)
    ctx.take_flags()
    for k, w in want.items():
        g = res[k]
        assert g.shape == w.shape, (k, g.shape, w.shape)
        it = torch.int32 if g.dtype == torch.float32 else torch.int64
        assert torch.equal(g.view(it), w.contiguous().view(it)), (entry, k)


def _bad_calls(ctx, dtype):
    """entry -> call(ls, ols, L, n) with valid device pointers for L <= 4 levels and n <= 8 columns (and beyond,
    so that a check that passed would still stay inside the allocations)."""
    lib, h = ctx.lib, ctx.handle
    dt = torch.float32 if dtype == np.float32 else torch.float64
    code = _lib._dtype_code(torch.empty(0, dtype=dt))
    buf = [torch.full((64, 64), 500.0, dtype=dt, device="cuda") for _ in range(8)]
    mask = torch.zeros((64, 64), dtype=torch.uint8, device="cuda")
    P = [b.data_ptr() for b in buf]
    arr = lambda k, at=1: (ctypes.c_void_p * k)(*P[at:at + k])                       # noqa: E731
    opts = _lib.make_options()
    pin = _lib.XpParcelIn(P[1], P[2], P[3])
    fo = _lib.XpIntersectionsOut(*P[2:8])
    zo = _lib.XpZeroAreasOut(*(P[2:7] + [mask.data_ptr()]))
    mo = _lib.XpMixedParcelOut(*P[2:8])
    s = ctx._stream()
    return {
        "moist_lapse": lambda ls, ols, L, n: lib.xp_moist_lapse(h, P[0], ls, L, n, code, P[1], P[2], P[3], ols, s),
        "parcel_profile": lambda ls, ols, L, n: lib.xp_parcel_profile(h, P[0], ls, L, n, code, ctypes.byref(pin),
                                                                      ctypes.byref(opts), P[4], P[5], ols, P[6], P[7],
                                                                      None, s),
        "lfc_el": lambda ls, ols, L, n: lib.xp_lfc_el(h, P[0], P[1], P[2], ls, L, n, code, P[3], P[4], P[5], P[6], P[7],
                                                      None, s),
        "cape_cin_base": lambda ls, ols, L, n: lib.xp_cape_cin_base(h, P[0], P[1], P[2], ls, L, n, code, P[3], P[4],
                                                                    ctypes.byref(opts), P[5], P[6], s),
        "interp_levels": lambda ls, ols, L, n: lib.xp_interp_levels(h, P[0], ls, 0, arr(1), arr(1, 5), 1, ls, L, n, code,
                                                                    None, 500.0, 1, s),
        "level_crossing": lambda ls, ols, L, n: lib.xp_level_crossing(h, P[0], ls, 0, P[1], ls, L, n, code, 273.15,
                                                                      P[2], s),
        "mixed_layer": lambda ls, ols, L, n: lib.xp_mixed_layer(h, P[0], ls, 0, arr(2), arr(2, 5), 1, -1, ls, L, n, code,
                                                                100.0, s),
        "mixed_parcel": lambda ls, ols, L, n: lib.xp_mixed_parcel(h, P[0], ls, 0, P[1], P[2], ls, L, n, code, 100.0,
                                                                  ctypes.byref(mo), s),
        "layer_bounds": lambda ls, ols, L, n: lib.xp_layer_bounds(h, P[0], ls, 0, L, n, code, 100.0, 1, P[1], P[2], s),
        "insert_level": lambda ls, ols, L, n: lib.xp_insert_level(h, P[0], ls, 0, P[1], arr(1, 2), arr(1, 3), arr(1, 5), 1, P[6],
                                                                  ls, ols, L, n, code, s),
        "shift_out_nans": lambda ls, ols, L, n: lib.xp_shift_out_nans(h, P[0], arr(1), arr(1, 5), 1,
                                                                      ls, L, n, code, None, s),
        "trapz": lambda ls, ols, L, n: lib.xp_trapz(h, P[0], ls, 0, arr(1), arr(1, 5), 1, ls, L, n, code, None, 0, 0, s),
        "find_intersections": lambda ls, ols, L, n: lib.xp_find_intersections(h, P[0], ls, 0, P[0], P[1], ls, ols, L, n,
                                                                              code, 1, ctypes.byref(fo), s),
        "trap_around_zeros": lambda ls, ols, L, n: lib.xp_trap_around_zeros(h, P[0], ls, 0, P[1], ls, ols, L, n, code,
                                                                            1, ctypes.byref(zo), s),
        "valid_data": lambda ls, ols, L, n: lib.xp_valid_data(h, P[0], ls, 0, L, n, code, s),
    }, (buf, mask)


BAD_ENTRIES = ["moist_lapse", "parcel_profile", "lfc_el", "cape_cin_base", "interp_levels", "level_crossing",
               "mixed_layer", "mixed_parcel", "layer_bounds", "insert_level", "shift_out_nans", "trapz",
               "find_intersections", "trap_around_zeros", "valid_data"]


@pytest.mark.parametrize("entry", BAD_ENTRIES)
def test_c_abi_rejects_strides_smaller_than_a_level(ctx, entry):
    """level_stride < n_columns, out_level_stride < n_columns, n_levels < 1 and n_columns < 0 are
    XP_ERR_INVALID_ARGUMENT with a message naming the entry; n_columns = 0 is XP_OK without a launch."""
    calls, keep = _bad_calls(ctx, np.float32)
    call = calls[entry]
    L, n = 4, 8
    assert call(n, n, L, n) == _lib.XP_OK                                 # the compact call is fine
    torch.cuda.synchronize()
    ctx.take_flags()
    bad = [(n - 1, n, L, n), (n, n, 0, n), (n, n, L, -1)]
    if entry in HAS_OUT_STRIDE:
        bad.append((n, n - 1, L, n))
    for args in bad:
        st = call(*args)
        assert st == 1, (entry, args, st)                                  # XP_ERR_INVALID_ARGUMENT
        msg = ctx.lib.xp_last_error(ctx.handle).decode()
        assert entry in msg, (entry, args, msg)
    before = ctx.launch_count()
    assert call(n, n, L, 0) == _lib.XP_OK
    assert ctx.launch_count() == before
    torch.cuda.synchronize()
    ctx.take_flags()


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_trap_around_zeros_mask_stays_compact_under_a_wide_output_stride(ctx, dtype):
    """xparcel.h: the mask is [n_levels][n_columns] whatever out_level_stride is."""
    dt = torch.float32 if dtype == np.float32 else torch.float64
    L, n, W = 12, 40, 57
    g = torch.Generator().manual_seed(3)
    x = torch.linspace(1000.0, 200.0, L, dtype=dt)[:, None].expand(L, n).contiguous().cuda()
    y = (torch.rand((L, n), generator=g, dtype=dt) - 0.5).cuda()
    outs = [torch.full((2 * L - 1, W), 5.0, dtype=dt, device="cuda") for _ in range(5)]
    mask = torch.full((L + 2, n), 7, dtype=torch.uint8, device="cuda")
    o = _lib.XpZeroAreasOut(*([t.data_ptr() for t in outs] + [mask.data_ptr()]))
    code = _lib._dtype_code(y)
    ctx._check(ctx.lib.xp_trap_around_zeros(ctx.handle, x.data_ptr(), n, 0, y.data_ptr(), n, W, L, n, code, 1,
                                            ctypes.byref(o), ctx._stream()), "xp_trap_around_zeros")
    areas, want = ctx.trap_around_zeros(x, y)
    assert torch.equal(mask[:L] != 0, want)
    assert bool((mask[L:] == 7).all())
    for t, k in zip(outs, _lib.ZERO_AREA_FIELDS):
        assert torch.equal(torch.nan_to_num(t[:, :n], nan=-1.0), torch.nan_to_num(areas[k], nan=-1.0)), k
        assert bool((t[:, n:] == 5.0).all()), k
