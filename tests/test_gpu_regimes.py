"""Every route of the fast kernels against the float64 oracle on real-world column regimes (tests/regime_columns.py):
high terrain, polar and plateau cold, tropical moist heat, surfaces above 1100 hPa, model tops at 3 and 0.01 hPa, 150
levels, and ERA5 pressure levels with the below-ground levels masked.

``launch_suite_fast`` picks its kernels from the call: a shared pressure axis takes the v7 sweep (default options) or
the generic sweep (other options), four launches; per-column pressure with two or three kinds and default options
takes the shared-memory adiabat table (``suite_fast_ptab_kernel``), three launches; per-column pressure otherwise
gathers the adiabats from the curve table (``suite_fast_pcol_kernel``), two launches; float64 columns on a shared axis
take ``launch_suite_fast_f64``, four launches.  The exact kernel is one launch.  Each test asserts the launch count, so
that it cannot silently test another kernel than the one it names.

What holds on every route and regime: NaN patterns identical to the oracle, ``level_shift`` bit-exact, ML/MU parcels
within float32 rounding, CAPE/CIN within ``FAST_BOUND`` of test_gpu_parity -- on the table route within the per-column
bound of ``table_allowance`` -- and the same against the float64 exact kernel on the same device buffers.  Columns
handed over to the float64 fix-up run the exact kernel's column code and match it bit for bit.
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

pytestmark = pytest.mark.gpu

FIELDS = list(FAST_BOUND)
KINDS = ("sb", "ml", "mu")
PROFILE_NAMES = ["pressure", "temperature", "virtual_temperature", "environment_temperature",
                 "environment_virtual_temperature", "environment_dewpoint"]
NON_DEFAULT = dict(virtual_temperature_correction=False, lcl_interp="linear", pos_cape_neg_cin=True)

# per-column pressure: case -> (regime, levels, model top [hPa], columns)
PCOL_CASES = {
    "terrain": ("terrain", 70, 20.0, 6000),
    "cold": ("cold", 70, 20.0, 6000),
    "moist_heat": ("moist_heat", 70, 20.0, 6000),
    "high_surface": ("high_surface", 70, 20.0, 6000),
    "above_1100": ("above_1100", 70, 20.0, 1500),
    "top3_L137": ("synth_like", 137, 3.0, 3000),
    "long_L150": ("synth_like", 150, 20.0, 3000),
    "top0.01_L137": ("synth_like", 137, 0.01, 2000),
    "top0.01_L150": ("synth_like", 150, 0.01, 2000),
}
# where the design hands every column over: a surface below the table's 1100 hPa, a level above its 2.5 hPa
ALL_HANDED_OVER = ("above_1100", "top0.01_L137", "top0.01_L150")
# the 37 shared ERA5 levels: case -> (regime, layout, columns)
AXIS_CASES = {
    "cold_era5": ("cold", "era5", 6000),
    "moist_heat_era5": ("moist_heat", "era5", 6000),
    "high_surface_era5": ("high_surface", "era5", 6000),
    "era5_masked": ("masked", "era5_masked", 6000),
}
# Ceiling of the fraction of columns handed over to the fix-up (last_exact_count / N) in the cases where only the
# uncertain columns are, with headroom over the largest fraction of any route measured on a B200 (1000 W) with these
# seeds (in the comment).  Cold parcels leave the table's adiabat range; high_surface includes its 15 % of columns
# above 1100 hPa; ERA5 masked below ground hands over every column whose lowest level is missing.
HANDOVER_CEILING = {
    "terrain": 0.03,             # 0.0143
    "cold": 0.20,                # 0.1498
    "moist_heat": 0.05,          # 0.0302
    "high_surface": 0.25,        # 0.1878
    "top3_L137": 0.025,          # 0.0120
    "long_L150": 0.05,           # 0.0320
    "cold_era5": 0.03,           # 0.0137
    "moist_heat_era5": 0.01,     # 0.0043
    "high_surface_era5": 0.03,   # 0.0143
    "era5_masked": 0.96,         # 0.9412
}

# max |table - reference evaluation| of the saturated parcel's virtual temperature [K] that test_ptab_accuracy holds
# the table to, per segment: (lowest pressure, highest pressure, error)
TABLE_ERROR = ((100.0, np.inf, 4e-4), (20.0, 100.0, 2.5e-3), (0.0, 20.0, 0.06))


def table_allowance(p_hi, p_lo):
    """Per-column CAPE/CIN allowance [J/kg] of the table route over the pressure range [p_lo, p_hi].

    The table route evaluates the saturated parcel's virtual temperature from the shared-memory table
    (fast::PTabView) instead of the reference's two curve nodes.  CAPE and CIN are Rd times the trapezoid integral of
    (Tv_parcel - Tv_env) over ln p, so an error of at most e_seg K in every row of a segment moves the integral by at
    most Rd * e_seg * (the segment's ln-p extent inside the integration range): clipping to the positive or negative
    part cannot make a difference larger than the difference itself, and the LFC / EL crossings that the error moves
    sit where the integrand is zero, so they add only second-order terms.  Summed over the segments of TABLE_ERROR:

        allowance = Rd * sum_seg e_seg * |ln p_hi - ln p_lo| restricted to the segment,

    with [p_lo, p_hi] = LFC..EL (EL missing: the column top) for CAPE and surface..LFC for CIN.  This is added to
    FAST_BOUND, which covers the float32 arithmetic that both per-column routes share."""
    tot = np.zeros(np.shape(p_hi))
    with np.errstate(invalid="ignore", divide="ignore"):
        for lo, hi, e in TABLE_ERROR:
            top = np.maximum(p_lo, lo)
            bot = np.minimum(p_hi, hi)
            tot += e * np.where(bot > top, np.log(bot / top), 0.0)
    return th.RD * np.nan_to_num(tot)


# --------------------------------------------------------------------------- fixtures
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


def _case_columns(case, seed_offset=0):
    """(p, T, Td, p0) of a case: float32 NumPy arrays."""
    if case in PCOL_CASES:
        regime, levels, top, n = PCOL_CASES[case]
        return rc.columns(regime, n, seed=100 + list(PCOL_CASES).index(case) + seed_offset, levels=levels, p_top=top)
    regime, layout, n = AXIS_CASES[case]
    return rc.columns(regime, n, seed=200 + list(AXIS_CASES).index(case) + seed_offset, layout=layout)


def _oracle(p, t, td, tables, opts=None, profile=False):
    """Flat dict of float64 [N] oracle outputs (``<kind>_<field>``, the ML/MU level shifts) and, with ``profile``,
    ``<kind>_profile``: the parcel_profile_with_lcl rows."""
    P, T, D = (np.asarray(x, np.float64) for x in (p, t, td))
    if P.ndim == 1:
        P = np.broadcast_to(P[:, None], T.shape)
    kw = dict(opts or {})
    compat = kw.pop("metpy_compat", "1.4.1")
    o = op.Options(op.MoistLapseLUT(tables), lcl_mode="converged", metpy_compat=compat)
    out = {}
    sb, sbp = op.surface_based_cape_cin(P, T, D, o, **kw)
    ml, mlp, mp = op.mixed_layer_cape_cin(P, T, D, o, depth=100, **kw)
    mu, mup, ul = op.most_unstable_cape_cin(P, T, D, o, depth=300, **kw)
    for kind, cc, prof in (("sb", sb, sbp), ("ml", ml, mlp), ("mu", mu, mup)):
        out[kind + "_cape"], out[kind + "_cin"] = cc["cape"], cc["cin"]
        for f in FIELDS[2:]:
            out[f"{kind}_{f}"] = prof[f]
        if profile:
            out[kind + "_profile"] = {k: prof[k] for k in PROFILE_NAMES}
    for k in ("pressure", "temperature", "dewpoint"):
        out["ml_parcel_" + k] = mp[k]
        out["mu_parcel_" + k] = ul[k]
    with np.errstate(invalid="ignore"):
        out["mu_level_shift"] = np.where(np.isnan(ul["pressure"]), P.shape[0], (P > ul["pressure"][None, :]).sum(0))
        out["ml_level_shift"] = np.where(np.isnan(P[0]), P.shape[0], (P >= (np.nanmax(P, axis=0) - 100.0)[None, :]).sum(0))
        valid = ~np.isnan(T)
        out["p_bottom"] = np.nanmax(np.where(valid, P, np.nan), axis=0)
        out["p_top"] = np.nanmin(np.where(valid, P, np.nan), axis=0)
    out["has_nan"] = bool(np.isnan(T).any() or np.isnan(D).any())
    return out


class Cache:
    """Inputs, oracle and exact-kernel results per (case, variant), computed once for the module."""

    def __init__(self, ctx, tables):
        self.ctx, self.tables, self.store = ctx, tables, {}

    def get(self, key, make):
        if key not in self.store:
            self.store[key] = make()
        return self.store[key]

    def inputs(self, case, q=False):
        def make():
            p, t, td, p0 = _case_columns(case)
            D = td
            if q:
                td = rc.specific_humidity(p, td)
                P = p.astype(np.float64) if p.ndim == 2 else np.broadcast_to(p.astype(np.float64)[:, None], t.shape)
                D = th.dewpoint_from_specific_humidity(P, t.astype(np.float64), td.astype(np.float64), "1.4.1")
            dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (p, t, td)]
            return dict(p=p, t=t, td=td, dew=D, p0=p0, dev=dev)
        return self.get(("in", case, q), make)

    def oracle(self, case, opts_name="default", q=False, profile=False):
        def make():
            x = self.inputs(case, q)
            return _oracle(x["p"], x["t"], x["dew"], self.tables, NON_DEFAULT if opts_name != "default" else None,
                           profile=profile)
        return self.get(("ora", case, opts_name, q, profile), make)

    def exact(self, case, kinds=KINDS, opts_name="default", q=False, profile=False, dtype=torch.float32):
        def make():
            x = self.inputs(case, q)
            o = dict(NON_DEFAULT) if opts_name != "default" else {}
            dev = [d.to(dtype) for d in x["dev"]]
            n0 = self.ctx.launch_count()
            r = self.ctx.cape_cin(*dev, kinds=kinds, options=_lib.make_options(exact_only=True, **o), profile=profile,
                                  specific_humidity=q)
            assert self.ctx.launch_count() == n0 + 1 and self.ctx.last_exact_count() == -1
            self.ctx.take_flags()
            return r
        return self.get(("exact", case, kinds, opts_name, q, profile, dtype), make)


@pytest.fixture(scope="module")
def cache(ctx, gpu_tables):
    return Cache(ctx, gpu_tables)


REPORT = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    """Per (case, route): the largest |CAPE - oracle| and |CIN - oracle| over the columns and the handed-over
    fraction; printed at the end of the module (pytest -s)."""
    yield REPORT
    if REPORT:
        print("\ncase / route                               max|dCAPE|  max|dCIN|  handed over")
        for k in sorted(REPORT):
            v = REPORT[k]
            print(f"{k:<42} {v['cape']:10.3g} {v['cin']:10.3g}  {v['frac']:.4f}")


def _run(ctx, dev, kinds, launches, **kw):
    """One fast call; asserts the number of kernel launches (which route ran).  Returns (results, handed over)."""
    n0 = ctx.launch_count()
    res = ctx.cape_cin(*dev, kinds=kinds, **kw)
    assert ctx.launch_count() - n0 == launches, f"{ctx.launch_count() - n0} launches, the route expects {launches}"
    n_exact = ctx.last_exact_count()
    assert n_exact >= 0
    ctx.take_flags()
    return res, n_exact


def _flat(res, kind):
    d = {f"{kind}_{f}": res[kind][f].double().cpu().numpy() for f in FIELDS}
    if kind != "sb":
        for f in ("pressure", "temperature", "dewpoint"):
            d[f"{kind}_parcel_{f}"] = res[kind]["parcel_" + f].double().cpu().numpy()
    return d


def _compare(res, ref, ora, kind, table=False, what=""):
    """res (GPU) against ref (oracle or exact kernel, flat dict) for one kind: NaN patterns identical, every field
    within FAST_BOUND (CAPE/CIN plus the per-column table allowance on the table route), the allowance inside the
    north star (0.1 % or 1 J/kg), ML/MU parcels within float32 rounding.  ``ora`` supplies the LFC / EL of the
    allowance.  Returns (max |dCAPE|, max |dCIN|)."""
    extra = {"cape": 0.0, "cin": 0.0}
    if table:
        lfc, el = ora[kind + "_lfc_pressure"], ora[kind + "_el_pressure"]
        has = ~np.isnan(lfc)
        extra["cape"] = np.where(has, table_allowance(lfc, np.where(np.isnan(el), ora["p_top"], el)), 0.0)
        extra["cin"] = np.where(has, table_allowance(ora["p_bottom"], lfc), 0.0)
    worst = {}
    for f in FIELDS:
        a = res[kind][f].double().cpu().numpy()
        b = ref[f"{kind}_{f}"]
        nan_mis = np.flatnonzero(np.isnan(a) != np.isnan(b))
        assert nan_mis.size == 0, f"{what}{kind}_{f}: NaN pattern differs in columns {nan_mis[:8]}"
        ok = ~np.isnan(b)
        bb = np.where(ok, b, 0.0)
        diff = np.where(ok, np.abs(a - bb), 0.0)
        rel, ab = FAST_BOUND[f]
        bound = rel * np.abs(bb) + ab + extra.get(f, 0.0)
        if f in ("cape", "cin"):
            inside = bound <= np.maximum(1.0, 1e-3 * np.abs(bb))
            assert inside.all(), (f"{what}{kind}_{f}: the bound leaves the north star in columns "
                                  f"{np.flatnonzero(~inside)[:8]}")
            worst[f] = float(diff.max()) if diff.size else 0.0
        over = np.flatnonzero(ok & (diff > bound))
        assert over.size == 0, (f"{what}{kind}_{f}: {over.size} columns outside the bound, e.g. "
                                f"{[(int(i), float(a[i]), float(b[i]), float(bound[i])) for i in over[:4]]}")
    if kind != "sb":
        for f in ("pressure", "temperature", "dewpoint"):
            a = res[kind]["parcel_" + f].double().cpu().numpy()
            b = ref[f"{kind}_parcel_{f}"]
            assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}{kind} parcel {f}: NaN pattern differs"
            ok = ~np.isnan(b)
            assert np.allclose(a[ok], b[ok], rtol=3e-7, atol=0), f"{what}{kind} parcel {f}"
    return worst["cape"], worst["cin"]


def _check_route(cache, case, res, n_exact, kinds, route, table=False, q=False, opts_name="default", dtype=torch.float32):
    """The whole comparison of one fast call: oracle, exact kernel, level shifts, hand-over count."""
    x = cache.inputs(case, q)
    n = x["t"].shape[1]
    ora = cache.oracle(case, opts_name, q)
    ex = cache.exact(case, KINDS, opts_name, q, dtype=dtype)
    dc = di = 0.0
    for kind in kinds:
        c, i = _compare(res, ora, ora, kind, table, what=f"{case}/{route} vs oracle: ")
        dc, di = max(dc, c), max(di, i)
        _compare(res, _flat(ex, kind), ora, kind, table, what=f"{case}/{route} vs exact: ")
        assert torch.equal(res[kind]["level_shift"], ex[kind]["level_shift"]), f"{case}/{route}: {kind} level_shift"
        if kind != "sb" and not ora["has_nan"]:
            assert np.array_equal(res[kind]["level_shift"].cpu().numpy(), ora[kind + "_level_shift"]), \
                f"{case}/{route}: {kind} level_shift differs from the oracle"
    frac = n_exact / n
    if case in ALL_HANDED_OVER:
        assert n_exact == n, f"{case}/{route}: {n_exact} of {n} columns handed over, the design hands over all"
    else:
        if case.startswith("high_surface") and x["p"].ndim == 2:
            n_above = int((x["p"][0] > 1100.0).sum())
            assert n_above > 0 and n_exact >= n_above, (case, route, n_exact, n_above)
        assert frac <= HANDOVER_CEILING[case], f"{case}/{route}: handed-over fraction {frac:.4f}"
    REPORT[f"{case} / {route}"] = dict(cape=dc, cin=di, frac=frac)


# --------------------------------------------------------------------------- per-column pressure, the table route
PAIRS = {"sb+ml": ("sb", "ml"), "sb+mu": ("sb", "mu"), "ml+mu": ("ml", "mu"), "all": KINDS}


@pytest.mark.parametrize("kinds", list(PAIRS))
@pytest.mark.parametrize("case", list(PCOL_CASES))
def test_table_route(ctx, cache, case, kinds):
    """suite_fast_ptab_kernel<K, false> (two or three kinds, default options, scalar outputs): K = 3, 5, 6, 7."""
    x = cache.inputs(case)
    res, n_exact = _run(ctx, x["dev"], PAIRS[kinds], 3)
    _check_route(cache, case, res, n_exact, PAIRS[kinds], f"table {kinds}", table=True)


# --------------------------------------------------------------------------- per-column pressure, the gather route
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("case", list(PCOL_CASES))
def test_gather_route(ctx, cache, case, kind):
    """suite_fast_pcol_kernel<K, 1, false> (one kind, default options): the adiabats gathered from the curve table."""
    x = cache.inputs(case)
    res, n_exact = _run(ctx, x["dev"], (kind,), 2)
    _check_route(cache, case, res, n_exact, (kind,), f"gather {kind}")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("case", ["terrain", "cold", "moist_heat", "high_surface", "top3_L137"])
def test_gather_route_profile_rows_other_options(ctx, cache, gpu_tables, case, kind):
    """suite_fast_pcol_kernel<K, 0, true> (run-time options, profile rows): scalars as on every route, and the
    parcel_profile_with_lcl rows against the oracle and the exact kernel."""
    x = cache.inputs(case)
    res, n_exact = _run(ctx, x["dev"], (kind,), 2, profile=True, options=_lib.make_options(**NON_DEFAULT))
    _check_route(cache, case, res, n_exact, (kind,), f"gather+profile {kind}", opts_name="other")
    prof = cache.oracle(case, "other", profile=True)[kind + "_profile"]
    ex = cache.exact(case, (kind,), "other", profile=True)[kind]
    n = prof["pressure"].shape[0]
    for k in PROFILE_NAMES:
        a = res[kind]["profile_" + k].double().cpu().numpy()
        e = ex["profile_" + k].double().cpu().numpy()
        b = prof[k]
        assert np.array_equal(np.isnan(a), np.isnan(e)), f"{case} {kind} {k}: NaN pattern differs from the exact kernel"
        assert np.array_equal(np.isnan(a[:n]), np.isnan(b)), f"{case} {kind} {k}: NaN pattern differs from the oracle"
        assert np.isnan(a[n:]).all()
        ok = ~np.isnan(b)
        assert np.allclose(a[:n][ok], b[ok], rtol=3e-6, atol=0), (case, kind, k, np.abs(a[:n][ok] - b[ok]).max())
        ok = ~np.isnan(e)
        assert np.allclose(a[ok], e[ok], rtol=3e-6, atol=0), (case, kind, k)


# --------------------------------------------------------------------------- specific humidity in place of the dewpoint
@pytest.mark.parametrize("route", ["table", "gather"])
@pytest.mark.parametrize("case", ["terrain", "cold", "moist_heat"])
def test_specific_humidity_routes(ctx, cache, case, route):
    """suite_fast_ptab_kernel<7, true> and suite_fast_pcol_kernel<K, 0, false, true>: q converted to the dewpoint on
    load, against the oracle lifting the float64 dewpoint of the same q."""
    x = cache.inputs(case, q=True)
    kinds, launches = (KINDS, 3) if route == "table" else (("mu",), 2)
    res, n_exact = _run(ctx, x["dev"], kinds, launches, specific_humidity=True)
    _check_route(cache, case, res, n_exact, kinds, f"q {route}", table=route == "table", q=True)


# --------------------------------------------------------------------------- the shared ERA5 axis
@pytest.mark.parametrize("variant", ["v7-f32", "generic-f32", "fast-f64"])
@pytest.mark.parametrize("case", list(AXIS_CASES))
def test_shared_axis(ctx, cache, case, variant):
    """suite_fast_kernel<K, 1, 640, 3> (float32, default options), the generic sweep MODE 0 (other options) and
    launch_suite_fast_f64 (float64 columns) on the 37 ERA5 levels."""
    x = cache.inputs(case)
    dtype = torch.float64 if variant == "fast-f64" else torch.float32
    opts_name = "other" if variant == "generic-f32" else "default"
    o = NON_DEFAULT if opts_name == "other" else {}
    res, n_exact = _run(ctx, [d.to(dtype) for d in x["dev"]], KINDS, 4, options=_lib.make_options(**o))
    assert res["sb"]["cape"].dtype == dtype
    _check_route(cache, case, res, n_exact, KINDS, variant, opts_name=opts_name, dtype=dtype)


# --------------------------------------------------------------------------- handed-over columns
@pytest.mark.parametrize("route", ["table", "gather"])
@pytest.mark.parametrize("case", list(ALL_HANDED_OVER))
def test_handed_over_columns_equal_the_exact_kernel(ctx, cache, case, route):
    """Where every column is handed over, the fix-up (suite_list_kernel<1>: pressure staged in shared memory, up to
    147 levels; suite_list_kernel<0> above) runs the exact kernel's float64 column code on the same columns: every
    output bit-identical."""
    x = cache.inputs(case)
    kinds, launches = (KINDS, 3) if route == "table" else (("ml",), 2)
    res, n_exact = _run(ctx, x["dev"], kinds, launches)
    assert n_exact == x["t"].shape[1]
    ex = cache.exact(case)
    for kind in kinds:
        for f in _lib.SCALAR_FIELDS:
            if kind == "sb" and f.startswith("parcel_"):
                continue
            assert torch.equal(res[kind][f].view(torch.int32), ex[kind][f].view(torch.int32)), (case, route, kind, f)
        assert torch.equal(res[kind]["level_shift"], ex[kind]["level_shift"])


# --------------------------------------------------------------------------- warp neighbours
N_MIXED = 40_013           # not a multiple of 32, 512 or 640


def _mixed_columns(layout):
    """N_MIXED columns, the regimes interleaved column by column so that every warp holds all of them.  Returns
    (p, T, Td, regime label [N]) as float32 NumPy arrays.  Per-column pressure: 70 levels; the masked columns are
    terrain columns whose lowest levels are missing, as pressure-level data below ground.  Shared axis: ERA5."""
    if layout == "model":
        names = ["terrain", "cold", "moist_heat", "high_surface", "terrain"]
    else:
        names = ["cold", "moist_heat", "high_surface", "synth_like", "masked"]
    m = len(names)
    per = -(-N_MIXED // m)
    parts = []
    for i, name in enumerate(names):
        lay = "model" if layout == "model" else ("era5_masked" if name == "masked" else "era5")
        p, t, td, _ = rc.columns(name, per, seed=300 + i, layout=lay)
        if layout == "model" and i == m - 1:
            k = np.random.default_rng(399).integers(1, 7, per)
            below = np.arange(t.shape[0])[:, None] < k[None, :]
            t[below] = np.nan
            td[below] = np.nan
        parts.append((p, t, td))
    label = np.arange(N_MIXED) % m
    idx = np.arange(N_MIXED) // m
    t = np.stack([parts[r][1][:, i] for r, i in zip(label, idx)], axis=1)
    td = np.stack([parts[r][2][:, i] for r, i in zip(label, idx)], axis=1)
    p = parts[0][0] if layout != "model" else np.stack([parts[r][0][:, i] for r, i in zip(label, idx)], axis=1)
    return p, t, td, label


MIXED_ROUTES = {
    # route: (layout, kinds, launches, call keywords, dtype)
    "table": ("model", KINDS, 3, {}, torch.float32),
    "gather": ("model", ("mu",), 2, {}, torch.float32),
    "gather-profile": ("model", ("ml",), 2, {"profile": True}, torch.float32),
    "v7-f32": ("era5", KINDS, 4, {}, torch.float32),
    "fast-f64": ("era5", KINDS, 4, {}, torch.float64),
}


@pytest.mark.parametrize("route", list(MIXED_ROUTES))
def test_warp_neighbours_do_not_move_results(ctx, route):
    """A column's result does not depend on the columns that share its warp or tile -- the warp-wide phase boundary
    of the v7 sweeps, tail lanes, the persistent tile loops.  The interleaved columns against (a) the same columns
    sorted by regime and (b) the slice from column 7, which regroups every warp: bit for bit."""
    layout, kinds, launches, kw, dtype = MIXED_ROUTES[route]
    p, t, td, label = _mixed_columns(layout)
    order = np.argsort(label, kind="stable")

    def run(cols):
        dev = [torch.from_numpy(np.ascontiguousarray(c)).cuda().to(dtype) for c in (p if p.ndim == 1 else cols[0],
                                                                                      cols[1], cols[2])]
        return _run(ctx, dev, kinds, launches, **kw)

    full, n_full = run((p, t, td))
    srt, n_srt = run((p[:, order] if p.ndim == 2 else p, t[:, order], td[:, order]))
    sl, _ = run((p[:, 7:] if p.ndim == 2 else p, t[:, 7:], td[:, 7:]))
    assert n_full == n_srt
    order_d = torch.from_numpy(order).cuda()
    fields = _lib.SCALAR_FIELDS + (_lib.PROFILE_FIELDS if kw.get("profile") else [])
    view = torch.int64 if dtype == torch.float64 else torch.int32
    for kind in kinds:
        for f in fields + ["level_shift"]:
            if kind == "sb" and f.startswith("parcel_"):
                continue
            a, b, c = full[kind][f], srt[kind][f], sl[kind][f]
            if a.is_floating_point():
                a, b, c = a.view(view), b.view(view), c.view(view)
            assert torch.equal(a[..., order_d], b), (route, kind, f, "sorted by regime")
            assert torch.equal(a[..., 7:], c), (route, kind, f, "slice from column 7")
