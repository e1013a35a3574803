"""Downdraft CAPE and the effective inflow layer on the GPU against their float64 oracles on the real-world column
regimes of tests/regime_columns.py: high terrain, polar cold, moist heat, surfaces above 1100 hPa, a 0.01 hPa model top
at 137 levels, ERA5 levels extrapolated or masked below ground, and short per-column and deep shared axes.

``launch_layer`` (xp_effective.cu) picks one of eight instantiations of ``effective_layer_kernel<T, AXIS, STAGED>`` at
run time from the occupancy the runtime reports: it stages a column in shared memory only when that costs no resident
CTA.  Each of the eight is named here by the shape that selects it on a B200, proven to have run by torch.profiler, and
compared with the oracle.  Staged and unstaged readers must give the same bits: padding a column with all-NaN levels
above its top moves it from one to the other and may change nothing but the padded levels' NaN outputs.

DCAPE's NaN set is pinned from the inputs alone (DESIGN.md 3.12): a column is NaN when it has no valid level, when its
lowest valid level is above 700 hPa and not ``isclose`` to it (it cannot bracket 700 hPa), or when a valid level lies
below 1100 hPa (the descent leaves the moist-adiabat table, which ends there).
"""

import re

import numpy as np
import pytest
import torch

import downdraft_oracle as dd
import effective_oracle as eo
import regime_columns as rc
from oracle import parcel as op
from oracle import tables as otab
from test_gpu_downdraft import _compare as dd_compare
from test_gpu_effective import _compare as eff_compare
from xarray_parcel_b200 import _lib

pytestmark = pytest.mark.gpu

DD_SCALARS = ["dcape", "downdraft_start_pressure", "downdraft_start_temperature"]
DD_PROFILE = "downdraft_parcel_temperature"
EFF_SCALARS = _lib.EFFECTIVE_FIELDS
EFF_LEVELS = _lib.EFFECTIVE_LEVEL_FIELDS
DTYPES = [torch.float32, torch.float64]
DTYPE_IDS = ["f32", "f64"]

# (id, regime, regime_columns.columns keywords): every regime on 70 model levels, on the 37 ERA5 levels
# extrapolated below ground and, where some surface lies below 1000 hPa, masked below ground; the 0.01 hPa top at 137
# levels; 40 and 24 per-column levels, which the staged per-column readers take.
CASES = [
    ("terrain", "terrain", {}),
    ("terrain_era5", "terrain", dict(layout="era5")),
    ("terrain_era5_masked", "terrain", dict(layout="era5_masked")),
    ("cold", "cold", {}),
    ("cold_era5", "cold", dict(layout="era5")),
    ("cold_era5_masked", "cold", dict(layout="era5_masked")),
    ("moist_heat", "moist_heat", {}),
    ("moist_heat_era5", "moist_heat", dict(layout="era5")),
    ("moist_heat_era5_masked", "moist_heat", dict(layout="era5_masked")),
    ("high_surface", "high_surface", {}),
    ("high_surface_era5", "high_surface", dict(layout="era5")),
    ("above_1100", "above_1100", {}),
    ("above_1100_era5", "above_1100", dict(layout="era5")),
    ("masked_era5_masked", "masked", dict(layout="era5_masked")),
    ("top_0.01hPa_L137", "synth_like", dict(levels=137, p_top=0.01)),
    ("terrain_L40", "terrain", dict(levels=40)),
    ("moist_heat_L24", "moist_heat", dict(levels=24)),
]
# shapes only the layer-kernel variant test reads, at N_COLUMNS / 2 columns (the deep axes' oracle is the slowest):
# deep shared axes and 16 per-column levels
AXIS_CASES = [
    ("axis_top_0.01hPa_L137", "synth_like", dict(layout="axis", levels=137, p_top=0.01)),
    ("axis_high_surface_L100", "high_surface", dict(layout="axis", levels=100, p_top=1.0)),
    ("terrain_L16", "terrain", dict(levels=16)),
]
N_COLUMNS = 1500
CASE_IDS = [c[0] for c in CASES]
ALL_IDS = CASE_IDS + [c[0] for c in AXIS_CASES]
STRIDED_CASE = "top_0.01hPa_L137"              # per-column pressure read through a level stride wider than N
ALLNAN_EVERY = 97                              # columns 5, 102, 199, ... are NaN on every level


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
    return np.asarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x, dtype=np.float64)


def _columns(regime, kw, n, seed):
    """float32 (p, T, Td) of a regime with every ALLNAN_EVERY-th column NaN on every level."""
    p, t, td, _ = rc.columns(regime, n, seed=seed, **kw)
    t[:, 5::ALLNAN_EVERY] = np.nan
    td[:, 5::ALLNAN_EVERY] = np.nan
    return p, t, td


class _Oracles:
    """Inputs and float64 oracle results per case, computed once: the float32 and float64 calls read the same values
    (the float32 inputs), so they share the oracle."""

    def __init__(self, tables):
        self.tables = tables
        self.cache = {}

    def inputs(self, case_id):
        i = ALL_IDS.index(case_id)
        _, regime, kw = (CASES + AXIS_CASES)[i]
        return _columns(regime, kw, N_COLUMNS if i < len(CASES) else N_COLUMNS // 2, seed=300 + i)

    def compat(self, case_id):
        return "1.4.1" if ALL_IDS.index(case_id) % 2 == 0 else "1.6.2"

    def get(self, case_id, which):
        key = (case_id, which)
        if key not in self.cache:
            P, T, D = [x.astype(np.float64) for x in self.inputs(case_id)]
            if which == "dd":
                opts = op.Options(op.MoistLapseLUT(self.tables), metpy_compat=self.compat(case_id))
                self.cache[key] = dd.downdraft_cape(P, T, D, opts)
            else:
                self.cache[key] = eo.effective_inflow_layer(P, T, D, op.Options(op.MoistLapseLUT(self.tables)))
        return self.cache[key]


@pytest.fixture(scope="module")
def oracles(gpu_tables):
    return _Oracles(gpu_tables)


def dcape_nan_rule(P, T, D):
    """The columns whose DCAPE is NaN, from the inputs alone: no valid level; the lowest valid level above 700 hPa and
    not isclose to it; a valid level below 1100 hPa (p > 1100), where the descent leaves the table."""
    p = np.broadcast_to(op._as2d(P), T.shape)
    valid = ~(np.isnan(p) | np.isnan(T) | np.isnan(D))
    lowest = np.where(valid, p, -np.inf).max(axis=0)
    no_bracket = (lowest < dd.BOTTOM) & ~dd._close(lowest, dd.BOTTOM)
    off_table = (valid & (p > 1100.0)).any(axis=0)
    return ~valid.any(axis=0) | no_bracket | off_table


def _rel_err(got, want):
    with np.errstate(invalid="ignore"):
        err = np.where(np.isnan(want), 0.0, np.abs(got - want) / np.maximum(np.abs(want), 1.0))
    return float(err.max()) if err.size else 0.0


def _kernels(fn):
    """Run ``fn`` under torch.profiler: (its result, {"gate": [...], "layer": [...]}) with the template arguments of
    every effective_gate_kernel / effective_layer_kernel launch the profiler recorded, e.g. "float, false, true"."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    seen = {"gate": [], "layer": []}
    for e in prof.events():
        m = re.search(r"effective_(gate|layer)_kernel<([^>]*)>", e.name)
        if m:
            seen[m.group(1)].append(m.group(2))
    return out, seen


def _to_gpu(arrays, dtype):
    return [torch.from_numpy(np.ascontiguousarray(x)).to(dtype).cuda() for x in arrays]


def _strided(p):
    """Per-column pressure [L, N] as a view with level stride N + 37."""
    n = p.shape[1]
    wide = torch.full((p.shape[0], n + 37), float("nan"), dtype=p.dtype, device=p.device)
    wide[:, :n] = p
    assert wide[:, :n].stride(0) == n + 37
    return wide[:, :n]


# ---- DCAPE on the regimes ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", CASE_IDS)
def test_dcape_regimes_against_oracle(ctx, gpu_tables, oracles, case, dtype):
    """Every regime x layout x dtype; metpy_compat 1.4.1 / 1.6.2 and the profile on / off alternate over the cases
    so that each dtype meets each combination; per-column pressure through a wide level stride on STRIDED_CASE."""
    i, j = CASE_IDS.index(case), DTYPES.index(dtype)
    p, t, td = oracles.inputs(case)
    P, T, D = [x.astype(np.float64) for x in (p, t, td)]
    ora = oracles.get(case, "dd")
    compat, profile = oracles.compat(case), (i + j) % 2 == 0
    pd, tt, tdv = _to_gpu((p, t, td), dtype)
    if case == STRIDED_CASE:
        pd = _strided(pd)
    got = ctx.downdraft_cape(pd, tt, tdv, metpy_compat=compat, profile=profile)
    assert (DD_PROFILE in got) == profile
    dd_compare(got, P, T, D, gpu_tables, compat=compat, float32=dtype == torch.float32, ora=ora)
    dcape = _np(got["dcape"])
    assert np.array_equal(np.isnan(dcape), dcape_nan_rule(P, T, D))
    print(f"REGIME_STAT dcape {case} {DTYPE_IDS[j]} compat={compat} profile={int(profile)} "
          f"max_rel_err={_rel_err(dcape, ora['dcape']):.2e} nan_fraction={np.isnan(dcape).mean():.4f}")


def test_dcape_nan_rule_is_reached_by_the_regimes(oracles):
    """Each branch of the NaN rule has columns here, so a kernel that turned one of them into numbers would fail the
    regime tests: surfaces above 700 hPa (terrain), below 1100 hPa (every above_1100 column), NaN levels below ground
    (masked ERA5) and columns that are NaN throughout."""
    def rule(case):
        P, T, D = [x.astype(np.float64) for x in oracles.inputs(case)]
        nan = dcape_nan_rule(P, T, D)
        return nan, nan[np.isfinite(T).any(axis=0)].mean()
    assert rule("above_1100")[0].all()
    assert 0.05 < rule("high_surface")[1] < 0.5
    assert 0.05 < rule("terrain")[1] < 0.6 and 0.05 < rule("terrain_era5_masked")[1] < 0.6
    for case in ("terrain_era5", "moist_heat"):                  # only the columns that are NaN throughout
        nan, frac = rule(case)
        assert frac == 0.0 and nan[5::ALLNAN_EVERY].all()


# ---- the effective inflow layer on the regimes ----------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("case", CASE_IDS)
def test_effective_regimes_against_oracle(ctx, gpu_tables, oracles, case, dtype):
    """Search and all-levels mode against the oracle; base and top bit-identical between the modes."""
    p, t, td = oracles.inputs(case)
    P, T, D = [x.astype(np.float64) for x in (p, t, td)]
    ora = oracles.get(case, "eff")
    f32 = dtype == torch.float32
    pd, tt, tdv = _to_gpu((p, t, td), dtype)
    if case == STRIDED_CASE:
        pd = _strided(pd)
    search = ctx.effective_inflow_layer(pd, tt, tdv)
    every = ctx.effective_inflow_layer(pd, tt, tdv, profile=True)
    for k in EFF_SCALARS:
        assert torch.equal(search[k].view(torch.int32 if f32 else torch.int64),
                           every[k].view(torch.int32 if f32 else torch.int64)), k
    eff_compare(search, P, T, D, gpu_tables, float32=f32, ora=ora)
    eff_compare(every, P, T, D, gpu_tables, float32=f32, ora=ora)
    cast = (lambda v: v.astype(np.float32).astype(np.float64)) if f32 else (lambda v: v)
    excuse = eo.valid_levels(P, T, D) & (T == D)
    err = max(_rel_err(np.where(excuse, np.nan, _np(every[k])), np.where(excuse, np.nan, cast(ora[k])))
              for k in EFF_LEVELS)
    with np.errstate(invalid="ignore"):
        tol = np.maximum(np.abs(ora["level_parcel_cape"]), 1.0) * 1e-6
        near = (np.abs(ora["level_parcel_cape"] - 100.0) < tol) | (np.abs(ora["level_parcel_cin"] + 250.0) < tol)
    base = _np(search["effective_inflow_base"])
    print(f"REGIME_STAT effective {case} {DTYPE_IDS[DTYPES.index(dtype)]} max_level_rel_err={err:.2e} "
          f"base_nan_fraction={np.isnan(base).mean():.4f} level_nan_fraction={np.isnan(_np(every[EFF_LEVELS[0]])).mean():.4f} "
          f"near_threshold_fraction={(near | excuse).any(axis=0).mean():.4f}")


# ---- every layer-kernel variant, by the shape that selects it ------------------------------------------------------

# (template arguments of effective_layer_kernel, case, dtype).  The occupancy rule: 3 CTAs of 128 threads per SM by
# registers, 228 KB of shared memory per SM (1 KB of it reserved per CTA).  A staged CTA holds 3 x L x 128 x sizeof(T)
# bytes on per-column pressure, 2 x L x 128 x sizeof(T) + 8 L bytes on a shared axis, and runs only where it keeps the
# 3 CTAs per SM of the unstaged kernel: up to 50 (float) / 25 (double) per-column levels, 74 / 37 shared levels.
VARIANTS = [
    ("float, true, true", "terrain_era5", torch.float32),             # 38 KB staged: 3 CTAs
    ("double, true, true", "terrain_era5", torch.float64),            # 74 KB staged: 3 CTAs
    ("float, true, false", "axis_top_0.01hPa_L137", torch.float32),   # 140 KB staged: 1 CTA
    ("double, true, false", "axis_high_surface_L100", torch.float64), # 201 KB staged: 1 CTA
    ("float, false, true", "terrain_L40", torch.float32),             # 60 KB staged: 3 CTAs
    ("double, false, true", "terrain_L16", torch.float64),            # 48 KB staged: 3 CTAs
    ("float, false, false", "terrain", torch.float32),                # 105 KB staged: 2 CTAs
    ("double, false, false", "terrain", torch.float64),               # 210 KB staged: 1 CTA
]


@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0].replace(", ", "_") for v in VARIANTS])
def test_each_layer_kernel_variant_runs_and_matches_the_oracle(ctx, gpu_tables, oracles, variant):
    name, case, dtype = variant
    gate = name.split(",")[0]
    p, t, td = oracles.inputs(case)
    P, T, D = [x.astype(np.float64) for x in (p, t, td)]
    pd, tt, tdv = _to_gpu((p, t, td), dtype)
    search, seen_s = _kernels(lambda: ctx.effective_inflow_layer(pd, tt, tdv))
    every, seen_a = _kernels(lambda: ctx.effective_inflow_layer(pd, tt, tdv, profile=True))
    print(f"REGIME_STAT variant {name}: L={T.shape[0]} {'shared' if P.ndim == 1 else 'per-column'} "
          f"search {seen_s} all-levels {seen_a}")
    assert seen_s == {"gate": [gate], "layer": [name]}, seen_s
    assert seen_a == {"gate": [gate], "layer": [name]}, seen_a
    f32 = dtype == torch.float32
    ora = oracles.get(case, "eff")
    eff_compare(search, P, T, D, gpu_tables, float32=f32, ora=ora)
    eff_compare(every, P, T, D, gpu_tables, float32=f32, ora=ora)
    for k in EFF_SCALARS:
        assert torch.equal(torch.nan_to_num(search[k], nan=-1.0), torch.nan_to_num(every[k], nan=-1.0)), k


# ---- staged and unstaged readers give the same bits -----------------------------------------------------------------

# (regime, keywords, dtype, levels after padding, layer kernel before, after)
PADDINGS = [
    ("terrain", dict(levels=40), torch.float32, 80, "float, false, true", "float, false, false"),
    ("terrain", dict(levels=16), torch.float64, 40, "double, false, true", "double, false, false"),
    ("masked", dict(layout="era5_masked"), torch.float32, 137, "float, true, true", "float, true, false"),
    ("terrain", dict(layout="era5"), torch.float64, 100, "double, true, true", "double, true, false"),
]


def _pad(x, levels):
    """``x`` [L, N] or [L] with all-NaN levels appended above its top up to ``levels``."""
    return torch.cat([x, torch.full((levels - x.shape[0],) + tuple(x.shape[1:]), float("nan"), dtype=x.dtype,
                                    device=x.device)]).contiguous()


@pytest.mark.parametrize("padding", PADDINGS, ids=[f"{v[0]}_{v[4].replace(', ', '_')}" for v in PADDINGS])
def test_padding_with_nan_levels_moves_staged_to_unstaged_and_keeps_the_bits(ctx, padding):
    regime, kw, dtype, levels, before, after = padding
    p, t, td = _to_gpu(_columns(regime, kw, 3000, seed=500 + PADDINGS.index(padding)), dtype)
    L = t.shape[0]
    pp, tp, tdp = _pad(p, levels), _pad(t, levels), _pad(td, levels)
    ints = torch.int32 if dtype == torch.float32 else torch.int64
    bits = lambda x: x.view(ints)                                                      # noqa: E731
    for profile in (False, True):
        ctx.take_flags()
        a, seen_a = _kernels(lambda: ctx.effective_inflow_layer(p, t, td, profile=profile))
        fa = ctx.take_flags()
        b, seen_b = _kernels(lambda: ctx.effective_inflow_layer(pp, tp, tdp, profile=profile))
        fb = ctx.take_flags()
        assert seen_a["layer"] == [before] and seen_b["layer"] == [after], (seen_a, seen_b)
        assert fa == fb
        for k in EFF_SCALARS:
            assert torch.equal(bits(a[k]), bits(b[k])), (k, profile)
        for k in (EFF_LEVELS if profile else []):
            assert torch.equal(bits(a[k]), bits(b[k][:L])), k
            assert bool(torch.isnan(b[k][L:]).all()), k
        assert 0.1 < float((~torch.isnan(a["effective_inflow_base"])).double().mean()) < 0.9
    # DCAPE, one kernel, must not see the padding either
    a = ctx.downdraft_cape(p, t, td, profile=True)
    b = ctx.downdraft_cape(pp, tp, tdp, profile=True)
    for k in DD_SCALARS:
        assert torch.equal(bits(a[k]), bits(b[k])), k
    assert torch.equal(bits(a[DD_PROFILE]), bits(b[DD_PROFILE][:L]))
    assert bool(torch.isnan(b[DD_PROFILE][L:]).all())
