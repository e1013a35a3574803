"""Downdraft CAPE on the GPU (xp_downdraft_cape and parcel_functions.downdraft_cape) against the NumPy restatement
of the contract (tests/downdraft_oracle.py): both dtypes, shared and per-column pressure, strided pressure, profile on
and off, NULL outputs, device and host inputs; determinism, column-permutation equivariance, 64-bit offsets and the
conv_properties keyword."""

import ctypes

import numpy as np
import pytest
import torch

import downdraft_oracle as dd
from oracle import parcel as op
from oracle import tables as otab
from oracle import thermo as th
from xarray_parcel_b200 import _lib, synth
import xarray_parcel_b200.parcel_functions as parcel

pytestmark = pytest.mark.gpu

SCALARS = ["dcape", "downdraft_start_pressure", "downdraft_start_temperature"]
PROFILE = "downdraft_parcel_temperature"


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


def _compare(got, P, T, D, tables, compat="1.4.1", float32=False, ora=None):
    """float64: the oracle at 1e-9; float32: the oracle fed the float32 inputs, rounded to float32, at 2 ulp.  ``ora``:
    the oracle's float64 result on these inputs and ``compat``, when the caller has it already."""
    if ora is None:
        ora = dd.downdraft_cape(P, T, D, op.Options(op.MoistLapseLUT(tables), metpy_compat=compat))
    if float32:
        ora = {k: v.astype(np.float32).astype(np.float64) for k, v in ora.items()}
    g = {k: _np(v) for k, v in got.items()}
    p2 = np.broadcast_to(op._as2d(P), T.shape)
    pmax = op.nanmax(np.where(np.isnan(T) | np.isnan(D), np.nan, p2))
    dd.assert_matches(g, ora, pmax, ora["downdraft_start_pressure"], rtol=2.4e-7 if float32 else 1e-9)
    return ora


def _columns(kind, n, seed):
    if kind == "shared":
        return synth.era5_columns(n, seed=seed, nan_columns=0.05, allnan_columns=0.01, saturated=0.1)
    return synth.model_level_columns(n, 70, seed=seed, nan_columns=0.05, allnan_columns=0.01, saturated=0.1)


@pytest.mark.parametrize("profile", [False, True], ids=["scalars", "profile"])
@pytest.mark.parametrize("pressure", ["shared", "per_column", "shared_strided", "per_column_strided"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_c_abi_against_oracle(ctx, gpu_tables, dtype, pressure, profile):
    n = 6000
    p, t, td = _columns(pressure.split("_strided")[0], n, seed=31)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    pd, tdv, tt = [x.to(dtype).cuda() for x in (p, td, t)]
    if pressure.endswith("strided"):
        if pd.dim() == 1:
            wide = torch.full((2 * pd.shape[0],), float("nan"), dtype=dtype, device="cuda")
            wide[::2] = pd
            pd = wide[::2]
        else:
            wide = torch.full((pd.shape[0], n + 37), float("nan"), dtype=dtype, device="cuda")
            wide[:, :n] = pd
            pd = wide[:, :n]
        assert pd.stride(0) != (1 if pd.dim() == 1 else n)
    compat = "1.6.2" if pressure.startswith("per_column") else "1.4.1"
    got = ctx.downdraft_cape(pd, tt, tdv, metpy_compat=compat, profile=profile)
    assert (PROFILE in got) == profile
    _compare(got, P, T, D, gpu_tables, compat=compat, float32=dtype == torch.float32)


def test_null_outputs_are_skipped(ctx):
    p, t, td = [x.cuda().double() for x in _columns("per_column", 3000, seed=32)]
    full = ctx.downdraft_cape(p, t, td, profile=True)
    for subset in (["dcape"], ["downdraft_start_pressure", PROFILE], ["downdraft_start_temperature"]):
        got = ctx.downdraft_cape(p, t, td, profile=True, outputs=subset)
        assert set(got) == set(subset)
        for k in subset:
            assert torch.equal(torch.nan_to_num(got[k], nan=-1.0), torch.nan_to_num(full[k], nan=-1.0)), k
    # every output NULL: nothing to do
    o = _lib.XpDowndraftOut(None, None, None, None, 0)
    st = ctx.lib.xp_downdraft_cape(ctx.handle, p.data_ptr(), p.stride(0), 0, t.data_ptr(), td.data_ptr(),
                                   t.stride(0), t.shape[0], t.shape[1], _lib.XP_F64, 141, ctypes.byref(o),
                                   ctx._stream())
    assert st == _lib.XP_OK


def test_c_abi_status_codes(ctx):
    p, t, td = [x.cuda() for x in _columns("shared", 100, seed=33)]
    out = torch.empty(100, device="cuda")
    o = _lib.XpDowndraftOut(out.data_ptr(), None, None, None, 0)

    def call(c, n=100, dtype=_lib.XP_F32, ls=100, compat=141, tp=t.data_ptr()):
        return c.lib.xp_downdraft_cape(c.handle, p.data_ptr(), 1, 1, tp, td.data_ptr(), ls, 37, n, dtype, compat,
                                       ctypes.byref(o), c._stream())

    assert call(ctx) == _lib.XP_OK
    assert call(ctx, n=0) == _lib.XP_OK
    assert call(ctx, dtype=7) == 1
    assert call(ctx, ls=50) == 1
    assert call(ctx, compat=150) == 1
    assert call(ctx, tp=None) == 1
    bare = _lib.Context(0)                                   # a context without tables
    try:
        assert call(bare) == 3                               # XP_ERR_TABLES_NOT_LOADED
        with pytest.raises(AssertionError, match="load_moist_adiabat_lookups"):
            bare.downdraft_cape(p, t, td)
    finally:
        bare.close()


def test_python_surface_numpy_torch_and_vert_axis(ctx, gpu_tables):
    p, t, td = _columns("per_column", 2000, seed=34)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    r = parcel.downdraft_cape(P, T, D, profile=True)
    assert isinstance(r["dcape"], np.ndarray) and r["dcape"].dtype == np.float64
    assert r.var_attrs["dcape"]["units"] == "J kg$^{-1}$" and "long_name" in r.var_attrs[PROFILE]
    ora = _compare(dict(r), P, T, D, gpu_tables)
    # vertical axis last, NumPy
    r2 = parcel.downdraft_cape(P.T.copy(), T.T.copy(), D.T.copy(), vert_axis=1, profile=True)
    for k in SCALARS:
        assert np.array_equal(r2[k], r[k], equal_nan=True)
    assert np.array_equal(r2[PROFILE].T, r[PROFILE], equal_nan=True)
    # CUDA tensors in, CUDA tensors out; float32 torch on the CPU comes back on the CPU
    r3 = parcel.downdraft_cape(torch.from_numpy(P).cuda(), torch.from_numpy(T).cuda(), torch.from_numpy(D).cuda())
    assert r3["dcape"].is_cuda and PROFILE not in r3
    assert np.array_equal(r3["dcape"].cpu().numpy(), r["dcape"], equal_nan=True)
    r4 = parcel.downdraft_cape(p, t, td, metpy_compat="1.6.2")
    assert not r4["dcape"].is_cuda and r4["dcape"].dtype == torch.float32
    _compare(dict(r4), P, T, D, gpu_tables, compat="1.6.2", float32=True)
    # a shared 1-D pressure axis as NumPy
    p1, t1, td1 = synth.era5_columns(2000, seed=35)
    r5 = parcel.downdraft_cape(p1.numpy().astype(np.float64), t1.numpy().astype(np.float64),
                               td1.numpy().astype(np.float64))
    _compare(dict(r5), p1.numpy().astype(np.float64), t1.numpy().astype(np.float64),
             td1.numpy().astype(np.float64), gpu_tables)
    assert np.isfinite(ora["dcape"]).mean() > 0.9


def test_deterministic_and_permutation_equivariant_at_era5_size(ctx):
    p, t, td = synth.era5_columns(3_114_720, seed=36, device="cuda", nan_columns=0.02)
    a = ctx.downdraft_cape(p, t, td, profile=True)
    b = ctx.downdraft_cape(p, t, td, profile=True)
    for k in a:
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k
    perm = torch.randperm(t.shape[1], device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    c = ctx.downdraft_cape(p, t[:, perm].contiguous(), td[:, perm].contiguous(), profile=True)
    for k in SCALARS:
        assert torch.equal(c[k].view(torch.int32), a[k][perm].view(torch.int32)), k
    assert torch.equal(c[PROFILE].view(torch.int32), a[PROFILE][:, perm].view(torch.int32))


def test_arrays_of_more_than_2_pow_32_elements(ctx, gpu_tables):
    """117 M ERA5 columns in one call: 4.33e9 elements in each input array and in the parcel-temperature profile,
    which the kernel writes on every level.  The field is a 1 M-column block repeated 117 times (2^32 is not a multiple
    of 10^6: a wrapped offset would land in a different column of the block), so every repetition must be
    bit-identical to the first; the last columns are checked against the oracle."""
    base_n, reps = 1_000_000, 117
    p, tb, tdb = synth.era5_columns(base_n, seed=37, device="cuda")
    L, n = tb.shape[0], base_n * reps
    assert L * n >= 2 ** 32
    t = torch.empty((L, n), dtype=torch.float32, device="cuda")
    td = torch.empty_like(t)
    t.view(L, reps, base_n).copy_(tb[:, None, :])
    td.view(L, reps, base_n).copy_(tdb[:, None, :])
    r = ctx.downdraft_cape(p, t, td, profile=True)
    del t, td
    for k in SCALARS:
        x = r[k].view(torch.int32).view(reps, base_n)
        assert bool((x == x[0:1]).all()), k
    x = r[PROFILE].view(torch.int32).view(L, reps, base_n)
    assert bool((x == x[:, 0:1]).all())
    tail = slice(n - 2000, n)
    got = {k: r[k][tail] for k in SCALARS}
    _compare(got, p.cpu().numpy().astype(np.float64), tb[:, base_n - 2000:].cpu().numpy().astype(np.float64),
             tdb[:, base_n - 2000:].cpu().numpy().astype(np.float64), gpu_tables, float32=True)
    del r, x
    torch.cuda.empty_cache()


def test_conv_properties_downdraft_keyword(ctx):
    p, t, td = synth.model_level_columns(3000, 60, seed=38, nan_columns=0.05, allnan_columns=0.0)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    q = th.saturation_mixing_ratio(P, D)
    q = q / (1 + q)
    H = 7500.0 * np.log(P[0][None, :] / P)
    dat = {"pressure": P, "temperature": T, "specific_humidity": q, "height_asl": H, "wind_u": H / 1000,
           "wind_v": -H / 2000, "wind_height_above_surface": H, "surface_wind_u": np.zeros(3000),
           "surface_wind_v": np.zeros(3000)}
    base = parcel.conv_properties(dict(dat))
    with_dd = parcel.conv_properties(dict(dat), downdraft=True)
    assert "dcape" not in base and set(with_dd) == set(base) | {"dcape"}
    for k in base:
        assert np.array_equal(np.asarray(with_dd[k]), np.asarray(base[k]), equal_nan=True), k
    td_gpu = parcel.dewpoint_from_specific_humidity(P, T, q)
    direct = parcel.downdraft_cape(P, T, td_gpu)["dcape"]
    masked = np.isnan(base["mixed_100_cape"])
    assert masked.any() and np.isnan(with_dd["dcape"][masked]).all()
    assert np.array_equal(with_dd["dcape"][~masked], direct[~masked], equal_nan=True)
    assert np.isfinite(with_dd["dcape"][~masked]).mean() > 0.9
