"""Storm kinematics and the effective-layer parameters on the GPU (xp_storm_kinematics,
xp_supercell_tornado_parameters and the parcel_functions surface) against the NumPy restatement of the contract
(tests/kinematics_oracle.py): both dtypes, level stride, NULL outputs, status codes, determinism, column permutation,
64-bit offsets, the effective composition on real-world regimes, NumPy / torch / xarray inputs and conv_properties."""

import ctypes

import numpy as np
import pytest
import torch

import kinematics_oracle as ko
import regime_columns as rc
from oracle import parcel as op
from oracle import tables as otab
from xarray_parcel_b200 import _lib
import xarray_parcel_b200.parcel_functions as parcel

pytestmark = pytest.mark.gpu

DEPTHS = (1000.0, 3000.0, 500.0, 6000.0)
INVALID = 1


@pytest.fixture(scope="module")
def ctx():
    c = _lib.get_context(0)
    if not c.tables_loaded():
        c.tables_build()
    return c


def _np(x):
    return np.asarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x, dtype=np.float64)


def _winds(regime, n, seed, layout="model"):
    p, t, td, p0 = rc.columns(regime, n, seed=seed, layout=layout)
    return rc.conv_fields(p, t, td, p0, seed=seed + 1)


def _layers(n, seed):
    rng = np.random.default_rng(seed)
    bot = rng.uniform(-400.0, 3000.0, n)
    top = bot + rng.uniform(-200.0, 5000.0, n)
    bot[::17] = np.nan
    top[3::29] = bot[3::29]
    return bot, top


def _compare(got, want, scale, float32):
    for k, w in want.items():
        g = _np(got[k])
        if float32:
            w = w.astype(np.float32).astype(np.float64)
        assert np.array_equal(np.isnan(g), np.isnan(w)), (k, np.flatnonzero(np.isnan(g) != np.isnan(w))[:5])
        tol = 1e-9 * scale[k] + (2.4e-7 * np.abs(np.nan_to_num(w)) if float32 else 0.0)
        bad = np.where(np.isnan(w), False, np.abs(g - w) > tol)
        assert not bad.any(), (k, np.flatnonzero(bad)[:5])


def _device(f, dtype, keys=("wind_height_above_surface", "wind_u", "wind_v", "surface_wind_u", "surface_wind_v")):
    return [torch.from_numpy(np.asarray(f[k])).to(dtype).cuda() for k in keys]


def _strided(x):
    L, n = x.shape
    wide = torch.full((L, n + 37), float("nan"), dtype=x.dtype, device=x.device)
    wide[:, :n] = x
    return wide[:, :n]


@pytest.mark.parametrize("strided", [False, True], ids=["contiguous", "strided"])
@pytest.mark.parametrize("mover", ["right", "left"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_c_abi_against_oracle(ctx, dtype, mover, strided):
    n = 800
    f = _winds("synth_like", n, seed=71)
    z, u, v, su, sv = _device(f, dtype)
    if strided:
        z, u, v = _strided(z), _strided(u), _strided(v)
        assert u.stride(0) == n + 37
    sl, bl = _layers(n, 72), _layers(n, 73)
    dev = lambda a: torch.from_numpy(a).to(dtype).cuda()                   # noqa: E731
    got = ctx.storm_kinematics(z, u, v, su, sv, mover=mover, depths=DEPTHS, srh_layer=(dev(sl[0]), dev(sl[1])),
                               bwd_layer=(dev(bl[0]), dev(bl[1])))
    assert all(x.dtype == dtype for x in got.values())
    Z, U, V, SU, SV = [x.cpu().double().numpy() for x in (z, u, v, su, sv)]
    SL = tuple(dev(x).cpu().double().numpy() for x in sl)
    BL = tuple(dev(x).cpu().double().numpy() for x in bl)
    want, scale = ko.storm_kinematics(Z, U, V, SU, SV, _lib.MOVERS[mover], DEPTHS, SL, BL)
    _compare(got, want, scale, dtype == torch.float32)
    assert np.isfinite(want["srh_0_3000m"]).mean() > 0.9


def test_null_outputs_are_skipped(ctx):
    f = _winds("terrain", 1500, seed=74, layout="era5")
    z, u, v, su, sv = _device(f, torch.float64)
    lay = tuple(torch.from_numpy(x).cuda() for x in _layers(1500, 75))
    full = ctx.storm_kinematics(z, u, v, su, sv, depths=DEPTHS, srh_layer=lay, bwd_layer=lay)
    for subset in (["bunkers_left_v"], ["srh_0_3000m", "bulk_wind_difference"], ["srh_layer", "mean_wind_u"],
                   ["srh_0_1000m"]):
        got = ctx.storm_kinematics(z, u, v, su, sv, depths=DEPTHS, srh_layer=lay, bwd_layer=lay, outputs=subset)
        assert set(got) == set(subset)
        for k in subset:
            assert torch.equal(torch.nan_to_num(got[k], nan=-1.0), torch.nan_to_num(full[k], nan=-1.0)), k
    comp = ctx.supercell_tornado_parameters(*[torch.rand(100, device="cuda", dtype=torch.float64) * 100
                                              for _ in range(6)])
    scp = ctx.supercell_tornado_parameters(*[torch.rand(100, device="cuda", dtype=torch.float64) for _ in range(6)],
                                           outputs=["supercell_composite_parameter"])
    assert set(comp) == set(_lib.COMPOSITE_FIELDS) and set(scp) == {"supercell_composite_parameter"}
    o = _lib.XpKinematicsOut()
    cols = _lib.XpWindColumns(z.data_ptr(), u.data_ptr(), v.data_ptr(), su.data_ptr(), sv.data_ptr(), 1500, 37,
                              _lib.XP_F64, 1500)
    kin = _lib.XpKinematicsIn(1, 0, (ctypes.c_double * 4)(), None, None, None, None)
    assert ctx.lib.xp_storm_kinematics(ctx.handle, ctypes.byref(cols), ctypes.byref(kin), ctypes.byref(o),
                                       ctx._stream()) == _lib.XP_OK


def test_c_abi_status_codes(ctx):
    n, L = 100, 20
    z = torch.rand((L, n), device="cuda") * 1000
    u, v = torch.rand_like(z), torch.rand_like(z)
    su, sv = u[0].clone(), v[0].clone()
    out = torch.empty(n, device="cuda")
    lay = torch.zeros(n, device="cuda")

    def call(cols_kw=None, in_kw=None, out_kw=None, c=ctx, null=None):
        cols = _lib.XpWindColumns(z.data_ptr(), u.data_ptr(), v.data_ptr(), su.data_ptr(), sv.data_ptr(), n, L,
                                  _lib.XP_F32, n)
        kin = _lib.XpKinematicsIn(1, 1, (ctypes.c_double * 4)(1000.0, 0, 0, 0), None, None, None, None)
        o = _lib.XpKinematicsOut()
        o.right_u = out.data_ptr()
        for obj, kw in ((cols, cols_kw), (kin, in_kw), (o, out_kw)):
            for k, val in (kw or {}).items():
                if k == "depths":
                    obj.depths = (ctypes.c_double * 4)(*val)
                elif k == "srh":
                    obj.srh = (ctypes.c_void_p * 4)(*val)
                else:
                    setattr(obj, k, val)
        args = [ctypes.byref(cols), ctypes.byref(kin), ctypes.byref(o)]
        if null is not None:
            args[null] = None
        return c.lib.xp_storm_kinematics(c.handle, *args, c._stream())

    assert call() == _lib.XP_OK
    assert call(cols_kw={"n_columns": 0}) == _lib.XP_OK
    for i in range(3):
        assert call(null=i) == INVALID
    for k in ("height", "wind_u", "wind_v", "surface_u", "surface_v"):
        assert call(cols_kw={k: None}) == INVALID, k
    assert call(cols_kw={"n_levels": 0}) == INVALID
    assert call(cols_kw={"level_stride": 50}) == INVALID
    assert call(cols_kw={"dtype": 7}) == INVALID
    assert call(in_kw={"mover": 0}) == INVALID and call(in_kw={"mover": 2}) == INVALID
    assert call(in_kw={"mover": -1}) == _lib.XP_OK
    assert call(in_kw={"n_depths": 5}) == INVALID and call(in_kw={"n_depths": -1}) == INVALID
    for bad in (0.0, -5.0, float("nan"), float("inf")):
        assert call(in_kw={"depths": (bad, 0, 0, 0)}) == INVALID, bad
    assert call(in_kw={"n_depths": 4, "depths": (1000.0, 2000.0, 3000.0, 4000.0)}) == _lib.XP_OK
    assert call(out_kw={"srh": (None, out.data_ptr(), None, None)}) == INVALID       # j >= n_depths
    assert call(in_kw={"srh_bottom": lay.data_ptr()}) == INVALID
    assert call(in_kw={"bwd_top": lay.data_ptr()}) == INVALID
    assert call(out_kw={"srh_layer": out.data_ptr()}) == INVALID
    assert call(out_kw={"bwd_magnitude": out.data_ptr()}) == INVALID
    assert call(in_kw={"bwd_bottom": lay.data_ptr(), "bwd_top": lay.data_ptr()},
                out_kw={"bwd_magnitude": out.data_ptr()}) == _lib.XP_OK
    p = [torch.rand(n, device="cuda") for _ in range(6)]
    f = ctx.lib.xp_supercell_tornado_parameters
    ptr = [x.data_ptr() for x in p]
    assert f(ctx.handle, *ptr, n, _lib.XP_F32, out.data_ptr(), out.data_ptr(), ctx._stream()) == _lib.XP_OK
    assert f(ctx.handle, *ptr, n, 7, out.data_ptr(), None, ctx._stream()) == INVALID
    assert f(ctx.handle, *ptr, -1, _lib.XP_F32, out.data_ptr(), None, ctx._stream()) == INVALID
    assert f(ctx.handle, None, *ptr[1:], n, _lib.XP_F32, out.data_ptr(), None, ctx._stream()) == INVALID
    assert f(ctx.handle, None, *ptr[1:], n, _lib.XP_F32, None, out.data_ptr(), ctx._stream()) == _lib.XP_OK
    assert f(ctx.handle, ptr[0], None, *ptr[2:], n, _lib.XP_F32, out.data_ptr(), None, ctx._stream()) == INVALID
    assert f(ctx.handle, *ptr[:5], None, n, _lib.XP_F32, None, out.data_ptr(), ctx._stream()) == INVALID
    assert f(ctx.handle, *ptr[:5], None, n, _lib.XP_F32, out.data_ptr(), None, ctx._stream()) == _lib.XP_OK


def test_composites_against_oracle(ctx):
    rng = np.random.default_rng(76)
    n = 100_000
    x = [rng.uniform(0, 5000, n), rng.uniform(-300, 600, n), rng.uniform(0, 40, n), rng.uniform(0, 4000, n),
         rng.uniform(-300, 0, n), rng.uniform(0, 3000, n)]
    for a in x:
        a[rng.random(n) < 0.02] = np.nan
    x[2][::97] = np.array([10.0, 20.0, 12.5, 30.0])[np.arange(x[2][::97].size) % 4]
    x[5][::89] = np.array([1000.0, 2000.0])[np.arange(x[5][::89].size) % 2]
    x[4][::83] = np.array([-50.0, -200.0])[np.arange(x[4][::83].size) % 2]
    want_scp = ko.supercell_composite(x[0], x[1], x[2])
    want_stp = ko.significant_tornado(x[3], x[1], x[2], x[5], x[4])
    for dtype in (torch.float64, torch.float32):
        xs = [torch.from_numpy(a).to(dtype).cuda() for a in x]
        got = ctx.supercell_tornado_parameters(*xs)
        X = [a.cpu().double().numpy() for a in xs]
        ws, wt = ko.supercell_composite(X[0], X[1], X[2]), ko.significant_tornado(X[3], X[1], X[2], X[5], X[4])
        if dtype == torch.float64:
            assert np.array_equal(ws, want_scp, equal_nan=True)
        cast = (lambda w: w.astype(np.float32).astype(np.float64)) if dtype == torch.float32 else (lambda w: w)
        assert np.array_equal(_np(got["supercell_composite_parameter"]), cast(ws), equal_nan=True)
        assert np.array_equal(_np(got["significant_tornado_parameter"]), cast(wt), equal_nan=True)


def test_deterministic_and_permutation_equivariant_at_era5_size(ctx):
    f = _winds("terrain", 20_000, seed=77, layout="era5")
    z, u, v, su, sv = _device(f, torch.float32)
    reps = 156                                                          # 3.12 M columns
    big = [x.repeat(1, reps) if x.dim() == 2 else x.repeat(reps) for x in (z, u, v, su, sv)]
    n = big[0].shape[1]
    lay = (torch.rand(n, device="cuda") * 2000 - 200, torch.rand(n, device="cuda") * 6000)
    kw = dict(depths=(1000.0, 3000.0), srh_layer=lay, bwd_layer=lay)
    a = ctx.storm_kinematics(*big, **kw)
    b = ctx.storm_kinematics(*big, **kw)
    for k in a:
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    pb = [x[:, perm].contiguous() if x.dim() == 2 else x[perm] for x in big]
    c = ctx.storm_kinematics(*pb, depths=(1000.0, 3000.0), srh_layer=(lay[0][perm], lay[1][perm]),
                             bwd_layer=(lay[0][perm], lay[1][perm]))
    for k in a:
        assert torch.equal(c[k].view(torch.int32), a[k][perm].view(torch.int32)), k
    assert float(torch.isfinite(a["srh_0_3000m"]).double().mean()) > 0.9


def test_one_call_over_more_than_2_pow_32_elements(ctx):
    """117 M columns of 37 levels in one call: 4.33e9 elements in each wind array.  The field is a 1 M-column block
    repeated 117 times (2^32 is not a multiple of 10^6: a wrapped offset would land in a different column of the
    block), so every repetition must be bit-identical to the first; the last columns are checked against the oracle."""
    base_n, reps = 1_000_000, 117
    L = 37
    rng = np.random.default_rng(78)
    zb = np.cumsum(rng.uniform(100.0, 800.0, (L, base_n)), axis=0) - rng.uniform(-200.0, 50.0, base_n)[None, :]
    ub = rng.normal(5.0, 8.0, (L, base_n)) + 0.003 * zb
    vb = rng.normal(0.0, 8.0, (L, base_n)) - 0.001 * zb
    sub, svb = rng.normal(0.0, 4.0, base_n), rng.normal(0.0, 4.0, base_n)
    n = base_n * reps
    assert L * n >= 2 ** 32
    big = []
    for a in (zb, ub, vb):
        x = torch.empty((L, n), dtype=torch.float32, device="cuda")
        x.view(L, reps, base_n).copy_(torch.from_numpy(a).float().cuda()[:, None, :])
        big.append(x)
    su = torch.from_numpy(sub).float().cuda().repeat(reps)
    sv = torch.from_numpy(svb).float().cuda().repeat(reps)
    r = ctx.storm_kinematics(*big, su, sv, depths=(1000.0, 3000.0))
    del big
    for k in r:
        x = r[k].view(torch.int32).view(reps, base_n)
        assert bool((x == x[0:1]).all()), k
    tail = slice(base_n - 500, base_n)
    args = [np.float32(a[:, tail]).astype(np.float64) for a in (zb, ub, vb)] + \
        [np.float32(a[tail]).astype(np.float64) for a in (sub, svb)]
    want, scale = ko.storm_kinematics(*args, 1, (1000.0, 3000.0))
    _compare({k: r[k][n - 500:] for k in r}, want, scale, float32=True)
    del r, x
    torch.cuda.empty_cache()


# ---- the effective composition ---------------------------------------------------------------------------------
def _gpu_tables(ctx):
    idx, cur = ctx.tables_get()
    pl, tl = otab.default_grids()
    return otab.AdiabatTables(pl, tl, idx, cur)


def _eff_inputs(layout, regime, n, seed):
    p, t, td, p0 = rc.columns(regime, n, seed=seed, layout=layout)
    f = rc.conv_fields(p, t, td, p0, seed=seed + 1)
    return p, f["temperature"], td, f


@pytest.mark.parametrize("mover", ["right", "left"])
@pytest.mark.parametrize("layout,regime", [("era5", "terrain"), ("era5_masked", "masked"), ("model", "synth_like"),
                                           ("model", "moist_heat")])
def test_effective_layer_parameters_against_oracle(ctx, layout, regime, mover):
    p, t, td, f = _eff_inputs(layout, regime, 3000, seed=80)
    P, T, D = [np.asarray(x, np.float64) for x in (p, t, td)]
    args = [f[k].astype(np.float64) for k in ("wind_height_above_surface", "wind_u", "wind_v", "surface_wind_u",
                                             "surface_wind_v")]
    H, U, V, SU, SV = args
    r = parcel.effective_layer_parameters(P, T, D, H, U, V, SU, SV, mover=mover)
    eff = parcel.effective_inflow_layer(P, T, D)
    for k in _lib.EFFECTIVE_FIELDS:
        assert np.array_equal(r[k], eff[k], equal_nan=True), k
    # the lift values the composition uses, from the library, composed by the oracle
    lifted = ctx.cape_cin(*[torch.from_numpy(x).cuda() for x in (P, T, D)], kinds=("ml", "mu"))
    ml, mu = [{k: _np(x) for k, x in lifted[kind].items()} for kind in ("ml", "mu")]
    pieces = {"effective_inflow_base": r["effective_inflow_base"], "effective_inflow_top": r["effective_inflow_top"],
              "mu_cape": mu["cape"], "mu_el_pressure": mu["el_pressure"], "ml_cape": ml["cape"], "ml_cin": ml["cin"],
              "ml_lcl_pressure": ml["lcl_pressure"]}
    opts = op.Options(op.MoistLapseLUT(_gpu_tables(ctx)))
    want, scale, extra = ko.effective_layer_parameters(P, T, D, H, U, V, SU, SV, opts, _lib.MOVERS[mover],
                                                       pieces=pieces)
    for k in ("effective_srh", "effective_bulk_wind_difference"):
        g, w = r[k], want[k]
        assert np.array_equal(np.isnan(g), np.isnan(w)), k
        bad = np.where(np.isnan(w), False, np.abs(g - w) > 1e-9 * scale[k])
        assert not bad.any(), (k, np.flatnonzero(bad)[:5])
    ebwd = want["effective_bulk_wind_difference"]
    with np.errstate(invalid="ignore"):
        edge = np.isclose(ebwd, 10.0, rtol=0, atol=1e-6) | np.isclose(ebwd, 12.5, rtol=0, atol=1e-6)
    for k in _lib.COMPOSITE_FIELDS:
        g, w = r[k], want[k]
        assert np.array_equal(np.isnan(g) | edge, np.isnan(w) | edge), k
        with np.errstate(invalid="ignore"):
            bad = ~edge & ~np.isnan(w) & (np.abs(g - w) > 1e-9 * (1.0 + np.abs(w)) * 100)
        assert not bad.any(), (k, np.flatnonzero(bad)[:5])
    has = ~np.isnan(r["effective_inflow_base"])
    assert has.mean() > 0.05
    assert np.isfinite(r["effective_srh"][has]).mean() > 0.9
    no = ~has & np.isfinite(pieces["mu_cape"])
    assert (r["supercell_composite_parameter"][no] == 0.0).all()
    assert (r["supercell_composite_parameter"][has] != 0).any()


def test_effective_layer_parameters_from_scratch_oracle(ctx):
    """The whole composition by the oracle (its own effective layer and lifts) on a small float64 sample."""
    p, t, td, f = _eff_inputs("model", "synth_like", 150, seed=82)
    P, T, D = [np.asarray(x, np.float64) for x in (p, t, td)]
    H, U, V, SU, SV = [f[k].astype(np.float64) for k in ("wind_height_above_surface", "wind_u", "wind_v",
                                                         "surface_wind_u", "surface_wind_v")]
    r = parcel.effective_layer_parameters(P, T, D, H, U, V, SU, SV)
    opts = op.Options(op.MoistLapseLUT(_gpu_tables(ctx)))
    want, scale, _ = ko.effective_layer_parameters(P, T, D, H, U, V, SU, SV, opts)
    same = np.isclose(r["effective_inflow_base"], want["effective_inflow_base"], rtol=0, atol=0, equal_nan=True) & \
        np.isclose(r["effective_inflow_top"], want["effective_inflow_top"], rtol=0, atol=0, equal_nan=True)
    assert same.mean() > 0.95
    for k in ("effective_srh", "effective_bulk_wind_difference") + tuple(_lib.COMPOSITE_FIELDS):
        g, w = r[k][same], want[k][same]
        assert np.array_equal(np.isnan(g), np.isnan(w)), k
        with np.errstate(invalid="ignore"):
            assert np.nanmax(np.abs(g - w) / (1.0 + np.abs(w))) < 1e-4, k


def test_python_surface_numpy_torch_vert_axis_and_xarray(ctx):
    import xr_double
    p, t, td, f = _eff_inputs("model", "synth_like", 1200, seed=84)
    P, T, D = [np.asarray(x, np.float64) for x in (p, t, td)]
    H, U, V, SU, SV = [f[k].astype(np.float64) for k in ("wind_height_above_surface", "wind_u", "wind_v",
                                                         "surface_wind_u", "surface_wind_v")]
    b = parcel.bunkers_storm_motion(SU, SV, U, V, H)
    assert isinstance(b["bunkers_right_u"], np.ndarray) and b.var_attrs["bunkers_right_u"]["units"] == "m s$^{-1}$"
    want, _ = ko.storm_kinematics(H, U, V, SU, SV, 1, (1000.0, 3000.0))
    for k in _lib.MOTION_FIELDS:
        assert np.allclose(b[k], want[k], rtol=1e-9, atol=1e-9, equal_nan=True), k
    s = parcel.storm_relative_helicity(SU, SV, U, V, H)
    assert set(s) == {"srh_0_1000m", "srh_0_3000m"} and "long_name" in s.var_attrs["srh_0_1000m"]
    assert np.allclose(s["srh_0_3000m"], want["srh_0_3000m"], rtol=1e-8, atol=1e-8, equal_nan=True)
    sl = parcel.storm_relative_helicity(SU, SV, U, V, H, depths=(250,), mover="left")
    assert set(sl) == {"srh_0_250m"}
    s2 = parcel.storm_relative_helicity(SU, SV, U.T.copy(), V.T.copy(), H.T.copy(), vert_axis=1)
    assert np.array_equal(s2["srh_0_1000m"], s["srh_0_1000m"], equal_nan=True)
    tt = [torch.from_numpy(x).cuda() for x in (SU, SV, U, V, H)]
    s3 = parcel.storm_relative_helicity(*tt)
    assert s3["srh_0_3000m"].is_cuda
    assert np.array_equal(s3["srh_0_3000m"].cpu().numpy(), s["srh_0_3000m"], equal_nan=True)
    s4 = parcel.bunkers_storm_motion(*[torch.from_numpy(x).float() for x in (SU, SV, U, V, H)])
    assert not s4["mean_wind_u"].is_cuda and s4["mean_wind_u"].dtype == torch.float32
    e = parcel.effective_layer_parameters(P, T, D, H, U, V, SU, SV)
    assert set(e) == set(_lib.EFFECTIVE_FIELDS) | set(_lib.EFFECTIVE_PARAMETER_FIELDS)
    assert e.var_attrs["effective_srh"]["units"] == "m$^{2}$ s$^{-2}$"
    et = parcel.effective_layer_parameters(*[torch.from_numpy(x).cuda() for x in (P, T, D, H, U, V, SU, SV)])
    for k in e:
        assert np.array_equal(et[k].cpu().numpy(), e[k], equal_nan=True), k
    scp = parcel.supercell_composite_parameter(np.array([2000.0, 1000.0]), np.array([100.0, 50.0]), 25.0)
    assert np.allclose(scp, [4.0, 1.0])
    stp = parcel.significant_tornado_parameter(np.array([1500.0]), 150.0, 25.0, 1500.0, -125.0)
    assert np.allclose(stp, [1.25 * 0.5 * 0.5])
    pf = xr_double.install()
    try:
        da = lambda a: xr_double.DataArray(a, dims=("model_level_number", "x"))    # noqa: E731
        sa = lambda a: xr_double.DataArray(a, dims=("x",))                          # noqa: E731
        rx = pf.storm_relative_helicity(sa(SU), sa(SV), da(U), da(V), da(H))
        assert np.array_equal(np.asarray(rx["srh_0_1000m"]), s["srh_0_1000m"], equal_nan=True)
        ex = pf.effective_layer_parameters(da(P), da(T), da(D), da(H), da(U), da(V), sa(SU), sa(SV))
        assert np.array_equal(np.asarray(ex["effective_srh"]), e["effective_srh"], equal_nan=True)
        assert ex["effective_srh"].attrs["units"] == "m$^{2}$ s$^{-2}$"
    finally:
        xr_double.uninstall()


@pytest.mark.parametrize("layout", ["model", "era5_masked"])
def test_conv_properties_kinematics_keyword(ctx, layout):
    p, t, td, f = _eff_inputs(layout, "masked" if layout == "era5_masked" else "synth_like", 2000, seed=86)
    dat = dict(f)
    base = parcel.conv_properties(dict(dat))
    kin = parcel.conv_properties(dict(dat), kinematics=True)
    new = set(_lib.MOTION_FIELDS) | {"srh_0_1000m", "srh_0_3000m"}
    assert set(kin) == set(base) | new and not new & set(base)
    for k in base:
        assert np.array_equal(np.asarray(kin[k]), np.asarray(base[k]), equal_nan=True), k
    eff = parcel.conv_properties(dict(dat), effective=True)
    both = parcel.conv_properties(dict(dat), effective=True, kinematics=True, mover="left")
    assert set(both) == set(eff) | new | set(_lib.EFFECTIVE_PARAMETER_FIELDS)
    for k in eff:
        assert np.array_equal(np.asarray(both[k]), np.asarray(eff[k]), equal_nan=True), k
    masked = np.isnan(base["mixed_100_cape"])
    direct = parcel.storm_relative_helicity(dat["surface_wind_u"], dat["surface_wind_v"], dat["wind_u"],
                                            dat["wind_v"], dat["wind_height_above_surface"])
    for k in ("srh_0_1000m", "srh_0_3000m"):
        assert np.isnan(kin[k][masked]).all()
        assert np.array_equal(kin[k][~masked], direct[k][~masked], equal_nan=True), k
    for k in _lib.EFFECTIVE_PARAMETER_FIELDS:
        assert np.isnan(both[k][masked]).all(), k
    assert np.isfinite(both["significant_tornado_parameter"][~masked]).mean() > 0.5
