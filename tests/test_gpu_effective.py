"""Effective inflow layer on the GPU (xp_effective_inflow_layer and parcel_functions.effective_inflow_layer) against
the NumPy restatement of the contract (tests/effective_oracle.py): both dtypes, shared, per-column and strided
pressure, search and all-levels modes, NULL outputs, status codes; the MU-level values against xp_cape_cin;
determinism, column-permutation equivariance, 64-bit offsets and the conv_properties keyword."""

import ctypes

import numpy as np
import pytest
import torch

import effective_oracle as eo
from oracle import parcel as op
from oracle import tables as otab
from oracle import thermo as th
from xarray_parcel_b200 import _lib, synth
import xarray_parcel_b200.parcel_functions as parcel

pytestmark = pytest.mark.gpu

SCALARS = _lib.EFFECTIVE_FIELDS
LEVELS = _lib.EFFECTIVE_LEVEL_FIELDS


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


def _compare(got, P, T, D, tables, float32=False, ora=None):
    """Levels: the oracle at 1e-9 (float64) or 2 ulp of float32 (the oracle fed the same float32 inputs), saturated
    starts excused.  Base / top: the search on the GPU's own level values where they were returned, and the oracle's
    base / top except in columns with a level value within the comparison tolerance of a threshold.  ``ora``: the
    oracle's float64 result on these inputs, when the caller has it already."""
    if ora is None:
        ora = eo.effective_inflow_layer(P, T, D, op.Options(op.MoistLapseLUT(tables)))
    g = {k: _np(v) for k, v in got.items()}
    valid = eo.valid_levels(P, T, D)
    rtol = 2.4e-7 if float32 else 1e-9
    excuse = valid & (T == D)
    for k in LEVELS:
        if k not in g:
            continue
        y = ora[k].astype(np.float32).astype(np.float64) if float32 else ora[k]
        assert np.array_equal(np.isnan(g[k]), np.isnan(y)), k
        with np.errstate(invalid="ignore"):
            err = np.where(np.isnan(y), 0.0, np.abs(g[k] - y) / np.maximum(np.abs(y), 1.0))
        assert not (err[~excuse] > rtol).any(), (k, np.nanmax(err[~excuse]))
    with np.errstate(invalid="ignore"):
        tol = np.maximum(np.abs(ora["level_parcel_cape"]), 1.0) * 1e-6
        near = (np.abs(ora["level_parcel_cape"] - 100.0) < tol) | (np.abs(ora["level_parcel_cin"] + 250.0) < tol)
    loose = (near | excuse).any(axis=0)
    for k in SCALARS:
        if k not in g:
            continue
        want = ora[k].astype(np.float32).astype(np.float64) if float32 else ora[k]
        same = np.isclose(g[k], want, rtol=0, atol=0, equal_nan=True)
        assert (same | loose).all(), (k, np.flatnonzero(~(same | loose))[:5])
    assert loose.mean() < 0.05
    return ora


def _columns(kind, n, seed):
    if kind == "shared":
        return synth.era5_columns(n, seed=seed, nan_columns=0.05, allnan_columns=0.01)
    return synth.model_level_columns(n, 70, seed=seed, nan_columns=0.05, allnan_columns=0.01)


def _strided(pd, n):
    if pd.dim() == 1:
        wide = torch.full((2 * pd.shape[0],), float("nan"), dtype=pd.dtype, device="cuda")
        wide[::2] = pd
        return wide[::2]
    wide = torch.full((pd.shape[0], n + 37), float("nan"), dtype=pd.dtype, device="cuda")
    wide[:, :n] = pd
    return wide[:, :n]


@pytest.mark.parametrize("profile", [False, True], ids=["search", "all_levels"])
@pytest.mark.parametrize("pressure", ["shared", "per_column", "shared_strided", "per_column_strided"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_c_abi_against_oracle(ctx, gpu_tables, dtype, pressure, profile):
    n = 1500 if pressure.startswith("shared") else 500
    p, t, td = _columns(pressure.split("_strided")[0], n, seed=51)
    pd, tt, tdv = [x.to(dtype).cuda() for x in (p, t, td)]
    P, T, D = [x.to(dtype).double().numpy() for x in (p, t, td)]
    if pressure.endswith("strided"):
        pd = _strided(pd, n)
        assert pd.stride(0) != (1 if pd.dim() == 1 else n)
    got = ctx.effective_inflow_layer(pd, tt, tdv, profile=profile)
    assert set(got) == set(SCALARS) | (set(LEVELS) if profile else set())
    _compare(got, P, T, D, gpu_tables, float32=dtype == torch.float32)
    if profile:
        g = {k: _np(v) for k, v in got.items()}
        valid = eo.valid_levels(P, T, D)
        gate = ~np.isnan(g["effective_inflow_base"])           # a passing gate always has a base: its own level
        base, top = eo.search(g["level_parcel_cape"], g["level_parcel_cin"], gate, valid)
        assert np.array_equal(eo.level_pressure(P, T.shape, base), g["effective_inflow_base"], equal_nan=True)
        assert np.array_equal(eo.level_pressure(P, T.shape, top), g["effective_inflow_top"], equal_nan=True)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", ["shared", "per_column"])
def test_search_and_all_levels_modes_agree_bitwise(ctx, dtype, kind):
    p, t, td = [x.to(dtype).cuda() for x in _columns(kind, 20000, seed=52)]
    a = ctx.effective_inflow_layer(p, t, td)
    b = ctx.effective_inflow_layer(p, t, td, profile=True)
    for k in SCALARS:
        assert torch.equal(torch.nan_to_num(a[k], nan=-1.0), torch.nan_to_num(b[k], nan=-1.0)), k
    assert 0.2 < float((~torch.isnan(a["effective_inflow_base"])).double().mean()) < 0.8


@pytest.mark.parametrize("kind", ["shared", "per_column"])
def test_level_values_at_the_mu_level_equal_xp_cape_cin(ctx, kind):
    """The lift from the most-unstable level IS the most-unstable lift: staging and the ln p table give the bits of
    the existing float64 column code."""
    for dtype in (torch.float32, torch.float64):
        p, t, td = [x.to(dtype).cuda() for x in _columns(kind, 30000, seed=53)]
        r = ctx.effective_inflow_layer(p, t, td, profile=True)
        mu = ctx.cape_cin(p, t, td, kinds=("mu",), options=_lib.make_options(exact_only=True))["mu"]
        k = mu["level_shift"].long()
        has = k < t.shape[0]
        cols = torch.arange(t.shape[1], device="cuda")[has]
        for name, f in (("level_parcel_cape", "cape"), ("level_parcel_cin", "cin")):
            got = r[name][k[has], cols]
            assert torch.equal(got, mu[f][has]), (name, dtype)


def test_null_outputs_are_skipped(ctx):
    p, t, td = [x.cuda().double() for x in _columns("per_column", 3000, seed=54)]
    full = ctx.effective_inflow_layer(p, t, td, profile=True)
    for subset in (["effective_inflow_base"], ["effective_inflow_top", "level_parcel_cin"], ["level_parcel_cape"]):
        got = ctx.effective_inflow_layer(p, t, td, profile=True, outputs=subset)
        assert set(got) == set(subset)
        for k in subset:
            assert torch.equal(torch.nan_to_num(got[k], nan=-1.0), torch.nan_to_num(full[k], nan=-1.0)), k
    cols, _, _ = ctx._columns(p, t, td)
    o = _lib.XpEffectiveOut(None, None, None, None, 0)
    st = ctx.lib.xp_effective_inflow_layer(ctx.handle, ctypes.byref(cols), None, 100.0, -250.0, ctypes.byref(o),
                                           ctx._stream())
    assert st == _lib.XP_OK


def test_c_abi_status_codes(ctx):
    p, t, td = [x.cuda() for x in _columns("shared", 100, seed=55)]
    out = torch.empty(100, device="cuda")
    o = _lib.XpEffectiveOut(out.data_ptr(), None, None, None, 0)

    def call(c, **changes):
        cols, _, _ = ctx._columns(p, t, td)
        for k, v in changes.items():
            setattr(cols, k, v)
        return c.lib.xp_effective_inflow_layer(c.handle, ctypes.byref(cols), None, 100.0, -250.0, ctypes.byref(o),
                                               c._stream())

    assert call(ctx) == _lib.XP_OK
    assert call(ctx, n_columns=0) == _lib.XP_OK
    assert call(ctx, mem=_lib.XP_MEM_HOST) == 1
    assert call(ctx, dewpoint_is_specific_humidity=1) == 1
    assert call(ctx, n_levels=0) == 1
    assert call(ctx, reserved_=1) == 1
    assert call(ctx, dtype=7) == 1
    assert call(ctx, level_stride=50) == 1
    lev = torch.empty((37, 100), device="cuda")
    o2 = _lib.XpEffectiveOut(None, None, lev.data_ptr(), None, 50)
    cols, _, _ = ctx._columns(p, t, td)
    assert ctx.lib.xp_effective_inflow_layer(ctx.handle, ctypes.byref(cols), None, 100.0, -250.0, ctypes.byref(o2),
                                             ctx._stream()) == 1
    bare = _lib.Context(0)                                   # a context without tables
    try:
        assert call(bare) == 3                               # XP_ERR_TABLES_NOT_LOADED
    finally:
        bare.close()


def test_python_surface_numpy_torch_vert_axis_and_xarray(ctx, gpu_tables):
    import xr_double
    p, t, td = _columns("per_column", 1000, seed=56)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    r = parcel.effective_inflow_layer(P, T, D, profile=True)
    assert isinstance(r["effective_inflow_base"], np.ndarray) and r["effective_inflow_base"].dtype == np.float64
    assert r.var_attrs["effective_inflow_base"]["units"] == "hPa" and "long_name" in r.var_attrs["level_parcel_cape"]
    _compare(dict(r), P, T, D, gpu_tables)
    r2 = parcel.effective_inflow_layer(P.T.copy(), T.T.copy(), D.T.copy(), vert_axis=1, profile=True)
    for k in SCALARS:
        assert np.array_equal(r2[k], r[k], equal_nan=True)
    assert np.array_equal(r2["level_parcel_cape"].T, r["level_parcel_cape"], equal_nan=True)
    r3 = parcel.effective_inflow_layer(torch.from_numpy(P).cuda(), torch.from_numpy(T).cuda(),
                                       torch.from_numpy(D).cuda())
    assert r3["effective_inflow_base"].is_cuda and "level_parcel_cape" not in r3
    assert np.array_equal(r3["effective_inflow_top"].cpu().numpy(), r["effective_inflow_top"], equal_nan=True)
    r4 = parcel.effective_inflow_layer(p, t, td)
    assert not r4["effective_inflow_base"].is_cuda and r4["effective_inflow_base"].dtype == torch.float32
    # non-default thresholds and options reach the kernel
    r5 = parcel.effective_inflow_layer(P, T, D, min_cape=1e9)
    assert np.isnan(r5["effective_inflow_base"]).all()
    r6 = parcel.effective_inflow_layer(P, T, D, profile=True, virtual_temperature_correction=False)
    assert not np.array_equal(r6["level_parcel_cape"], r["level_parcel_cape"], equal_nan=True)
    # xarray (the test double)
    pf = xr_double.install()
    try:
        da = lambda a: xr_double.DataArray(a, dims=("model_level_number", "x"))
        rx = pf.effective_inflow_layer(da(P), da(T), da(D))
        assert np.array_equal(np.asarray(rx["effective_inflow_base"]), r["effective_inflow_base"], equal_nan=True)
        assert rx["effective_inflow_top"].attrs["units"] == "hPa"
    finally:
        xr_double.uninstall()


def test_pressures_not_unique_is_raised(ctx):
    p, t, td = _columns("per_column", 200, seed=57)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    P[1, 5] = P[0, 5]                                        # a repeated pressure at the surface of one column ...
    T[:2, 5] = D[:2, 5] = T[0, 5] + 10.0                     # ... where the most-unstable parcel is
    with pytest.raises(AssertionError, match="not unique"):
        parcel.effective_inflow_layer(P, T, D)


def test_deterministic_and_permutation_equivariant_at_era5_size(ctx):
    p, t, td = synth.era5_columns(3_114_720, seed=58, device="cuda", nan_columns=0.02)
    a = ctx.effective_inflow_layer(p, t, td)
    b = ctx.effective_inflow_layer(p, t, td)
    for k in a:
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k
    perm = torch.randperm(t.shape[1], device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    c = ctx.effective_inflow_layer(p, t[:, perm].contiguous(), td[:, perm].contiguous())
    for k in SCALARS:
        assert torch.equal(c[k].view(torch.int32), a[k][perm].view(torch.int32)), k


def test_all_levels_over_more_than_2_pow_32_elements(ctx, gpu_tables):
    """117 M ERA5 columns in one all-levels call: 4.33e9 elements in each input array and in each level output.  The
    field is a 1 M-column block repeated 117 times (2^32 is not a multiple of 10^6: a wrapped offset would land in a
    different column of the block), so every repetition must be bit-identical to the first; the last columns are
    checked against the oracle."""
    base_n, reps = 1_000_000, 117
    p, tb, tdb = synth.era5_columns(base_n, seed=59, device="cuda")
    L, n = tb.shape[0], base_n * reps
    assert L * n >= 2 ** 32
    t = torch.empty((L, n), dtype=torch.float32, device="cuda")
    td = torch.empty_like(t)
    t.view(L, reps, base_n).copy_(tb[:, None, :])
    td.view(L, reps, base_n).copy_(tdb[:, None, :])
    r = ctx.effective_inflow_layer(p, t, td, profile=True)
    del t, td
    for k in SCALARS:
        x = r[k].view(torch.int32).view(reps, base_n)
        assert bool((x == x[0:1]).all()), k
    for k in LEVELS:
        x = r[k].view(torch.int32).view(L, reps, base_n)
        assert bool((x == x[:, 0:1]).all()), k
    tail = slice(n - 1000, n)
    got = {k: r[k][tail] for k in SCALARS}
    got.update({k: r[k][:, tail] for k in LEVELS})
    _compare(got, p.cpu().double().numpy(), tb[:, base_n - 1000:].cpu().double().numpy(),
             tdb[:, base_n - 1000:].cpu().double().numpy(), gpu_tables, float32=True)
    del r, x
    torch.cuda.empty_cache()


def test_conv_properties_effective_keyword(ctx):
    p, t, td = synth.model_level_columns(2000, 60, seed=60, nan_columns=0.05, allnan_columns=0.0)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    q = th.saturation_mixing_ratio(P, D)
    q = q / (1 + q)
    H = 7500.0 * np.log(P[0][None, :] / P)
    dat = {"pressure": P, "temperature": T, "specific_humidity": q, "height_asl": H, "wind_u": H / 1000,
           "wind_v": -H / 2000, "wind_height_above_surface": H, "surface_wind_u": np.zeros(2000),
           "surface_wind_v": np.zeros(2000)}
    base = parcel.conv_properties(dict(dat))
    with_eff = parcel.conv_properties(dict(dat), effective=True)
    assert set(with_eff) == set(base) | set(SCALARS) and not set(SCALARS) & set(base)
    for k in base:
        assert np.array_equal(np.asarray(with_eff[k]), np.asarray(base[k]), equal_nan=True), k
    td_gpu = parcel.dewpoint_from_specific_humidity(P, T, q)
    direct = parcel.effective_inflow_layer(P, T, td_gpu)
    masked = np.isnan(base["mixed_100_cape"])
    assert masked.any()
    for k in SCALARS:
        assert np.isnan(with_eff[k][masked]).all()
        assert np.array_equal(with_eff[k][~masked], np.asarray(direct[k])[~masked], equal_nan=True), k
    assert np.isfinite(with_eff["effective_inflow_base"][~masked]).mean() > 0.1
