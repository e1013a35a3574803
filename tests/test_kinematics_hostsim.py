"""Storm kinematics and the supercell / tornado composites: the column code of xp_kinematics.cuh (host-compiled from
tests/hostsim/hostsim_kinematics.cpp) against known answers, invariances and the NumPy restatement of the contract
(tests/kinematics_oracle.py, DESIGN.md section 3.14) on synthetic, real-world-regime and hand-built columns."""

import numpy as np
import pytest

import hostsim_kinematics as hs
import kinematics_oracle as ko
import regime_columns as rc

MOTION = ["bunkers_right_u", "bunkers_right_v", "bunkers_left_u", "bunkers_left_v", "mean_wind_u", "mean_wind_v"]
DEPTHS = (1000.0, 3000.0, 500.0, 6000.0)
BWD = ["bulk_wind_difference_u", "bulk_wind_difference_v", "bulk_wind_difference"]


def _check(z, u, v, su, sv, mover=1, depths=DEPTHS, srh_layer=None, bwd_layer=None, motion=True):
    """Host build against the oracle: |got - oracle| <= 1e-9 (1 + sum |terms|) and identical NaN patterns.  Returns
    (host result, oracle result)."""
    got = hs.storm_kinematics(z, u, v, su, sv, mover, depths, srh_layer, bwd_layer, motion)
    want, scale = ko.storm_kinematics(z, u, v, su, sv, mover, depths, srh_layer, bwd_layer, motion)
    for k, w in want.items():
        g = got[k]
        assert np.array_equal(np.isnan(g), np.isnan(w)), (k, np.flatnonzero(np.isnan(g) != np.isnan(w))[:5])
        err = np.where(np.isnan(w), 0.0, np.abs(g - w) / scale[k])
        assert not (err > 1e-9).any(), (k, float(err.max()))
    return got, want


def _sheared(n, L, seed, nan_levels=0.0):
    """Irregular AGL levels up to 12-16 km with seeded veering / backing shear and noise."""
    rng = np.random.default_rng(seed)
    dz = rng.uniform(50.0, 900.0, (L, n))
    z = np.cumsum(dz, axis=0) - rng.uniform(-300.0, 40.0, n)[None, :]          # some levels below ground
    km = np.clip(z, 0.0, None) / 1000.0
    turn = rng.uniform(-0.4, 0.4, n)[None, :] * km
    speed = rng.uniform(0.0, 6.0, n)[None, :] * km + rng.normal(0.0, 3.0, n)[None, :]
    u = speed * np.cos(turn) + rng.normal(0.0, 1.0, (L, n))
    v = speed * np.sin(turn) + rng.normal(0.0, 1.0, (L, n))
    if nan_levels:
        hole = rng.random((L, n)) < nan_levels
        which = rng.integers(0, 3, (L, n))
        z[hole & (which == 0)] = np.nan
        u[hole & (which == 1)] = np.nan
        v[hole & (which == 2)] = np.nan
    return z, u, v, rng.normal(0.0, 4.0, n), rng.normal(0.0, 4.0, n)


def _layers(n, seed):
    rng = np.random.default_rng(seed)
    bot = rng.uniform(-400.0, 3000.0, n)
    top = bot + rng.uniform(-200.0, 5000.0, n)
    bot[::17] = np.nan
    top[5::23] = np.nan
    top[3::29] = bot[3::29]                                         # zero depth
    return bot, top


# ---- known answers (independent of the oracle) ------------------------------------------------------------------
def _straight_line(seed=0):
    rng = np.random.default_rng(seed)
    z = np.concatenate([[0.0], np.sort(rng.uniform(10.0, 12000.0, 40)), [500.0, 3000.0, 5500.0, 6000.0]])
    z = np.unique(z)
    z = z[z > 0][:, None]
    return z, 0.01 * z, np.zeros_like(z), np.zeros(1), np.zeros(1)


@pytest.mark.parametrize("impl", ["hostsim", "oracle"])
def test_straight_line_shear_known_answers(impl):
    z, u, v, su, sv = _straight_line()
    for mover, srh3 in ((1, 225.0), (-1, -225.0)):
        if impl == "hostsim":
            r = hs.storm_kinematics(z, u, v, su, sv, mover, (3000.0,))
        else:
            r, _ = ko.storm_kinematics(z, u, v, su, sv, mover, (3000.0,))
        assert np.allclose([r[k][0] for k in MOTION], [30.0, -7.5, 30.0, 7.5, 30.0, 0.0], rtol=0, atol=1e-12)
        assert abs(r["srh_0_3000m"][0] - srh3) < 1e-10


def test_uniform_wind_has_no_bunkers_motion():
    z = np.arange(250.0, 9001.0, 250.0)[:, None]
    u, v = np.full_like(z, 10.0), np.full_like(z, -5.0)
    r = hs.storm_kinematics(z, u, v, [10.0], [-5.0], 1, (1000.0,))
    assert all(np.isnan(r[k][0]) for k in MOTION) and np.isnan(r["srh_0_1000m"][0])
    r, _ = ko.storm_kinematics(z, u, v, [10.0], [-5.0], 1, (1000.0,))
    assert all(np.isnan(r[k][0]) for k in MOTION)


# ---- invariances --------------------------------------------------------------------------------------------------
def _run(z, u, v, su, sv, mover=1, lay=None):
    return hs.storm_kinematics(z, u, v, su, sv, mover, (1000.0, 3000.0), srh_layer=lay, bwd_layer=lay)


def _close(a, b, atol):
    return np.allclose(a, b, rtol=0, atol=atol, equal_nan=True)


def test_constant_wind_shift():
    z, u, v, su, sv = _sheared(400, 40, seed=1)
    lay = _layers(400, 2)
    a = _run(z, u, v, su, sv, lay=lay)
    b = _run(z, u + 7.25, v - 3.5, su + 7.25, sv - 3.5, lay=lay)
    for k, d in (("bunkers_right_u", 7.25), ("bunkers_left_u", 7.25), ("mean_wind_u", 7.25),
                 ("bunkers_right_v", -3.5), ("bunkers_left_v", -3.5), ("mean_wind_v", -3.5)):
        assert _close(b[k], a[k] + d, 1e-9), k
    for k in ["srh_0_1000m", "srh_0_3000m", "srh_layer"] + BWD:
        assert _close(b[k], a[k], 1e-8), k
    assert np.isfinite(a["srh_0_3000m"]).mean() > 0.5


def test_rotation():
    z, u, v, su, sv = _sheared(400, 40, seed=3)
    lay = _layers(400, 4)
    th = 0.7
    c, s = np.cos(th), np.sin(th)
    rot = lambda x, y: (c * x - s * y, s * x + c * y)                       # noqa: E731
    a = _run(z, u, v, su, sv, lay=lay)
    b = _run(z, *rot(u, v), *rot(su, sv), lay=lay)
    for pre in ("bunkers_right", "bunkers_left", "mean_wind"):
        ru, rv = rot(a[pre + "_u"], a[pre + "_v"])
        assert _close(b[pre + "_u"], ru, 1e-9) and _close(b[pre + "_v"], rv, 1e-9), pre
    for k in ("srh_0_1000m", "srh_0_3000m", "srh_layer", "bulk_wind_difference"):
        assert _close(b[k], a[k], 1e-8), k


def test_mirror_swaps_movers():
    z, u, v, su, sv = _sheared(400, 40, seed=5)
    lay = _layers(400, 6)
    right = _run(z, u, v, su, sv, 1, lay)
    left = _run(z, u, v, su, sv, -1, lay)
    m = _run(z, u, -v, su, -sv, 1, lay)
    assert _close(m["bunkers_right_u"], right["bunkers_left_u"], 1e-9)
    assert _close(m["bunkers_right_v"], -right["bunkers_left_v"], 1e-9)
    assert _close(m["bunkers_left_u"], right["bunkers_right_u"], 1e-9)
    for k in ("srh_0_1000m", "srh_0_3000m", "srh_layer"):
        assert _close(m[k], -left[k], 1e-8), k


def test_level_on_the_interpolant_changes_nothing():
    z, u, v, su, sv = _sheared(300, 40, seed=7)
    lay = _layers(300, 8)
    a = _run(z, u, v, su, sv, lay=lay)
    k = 12                                                                  # a level between k and k + 1
    f = 0.37
    zi = z[k] + f * (z[k + 1] - z[k])
    ui = u[k] + (zi - z[k]) * (u[k + 1] - u[k]) / (z[k + 1] - z[k])
    vi = v[k] + (zi - z[k]) * (v[k + 1] - v[k]) / (z[k + 1] - z[k])
    ins = lambda x, y: np.concatenate([x[:k + 1], y[None, :], x[k + 1:]])   # noqa: E731
    b = _run(ins(z, zi), ins(u, ui), ins(v, vi), su, sv, lay=lay)
    for key in a:
        if key != "levels_read":
            assert _close(b[key], a[key], 1e-8), key


# ---- against the oracle ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mover", [1, -1], ids=["right", "left"])
@pytest.mark.parametrize("nan_levels", [0.0, 0.08])
def test_synthetic_columns_against_oracle(mover, nan_levels):
    z, u, v, su, sv = _sheared(600, 45, seed=11, nan_levels=nan_levels)
    su[::41] = np.nan
    got, want = _check(z, u, v, su, sv, mover, srh_layer=_layers(600, 12), bwd_layer=_layers(600, 13))
    assert np.isfinite(want["srh_0_3000m"]).mean() > 0.5 and np.isfinite(want["srh_layer"]).mean() > 0.3


@pytest.mark.parametrize("layout,regime", [("model", "synth_like"), ("era5", "terrain"), ("era5_masked", "masked"),
                                           ("model", "high_surface")])
def test_regime_columns_against_oracle(layout, regime):
    p, t, td, p0 = rc.columns(regime, 500, seed=21, layout=layout)
    f = rc.conv_fields(p, t, td, p0, seed=22)
    z, u, v = f["wind_height_above_surface"], f["wind_u"], f["wind_v"]
    assert (z < 0).any() or layout == "model"
    for dtype in (np.float64, np.float32):
        args = [x.astype(dtype).astype(np.float64) for x in (z, u, v, f["surface_wind_u"], f["surface_wind_v"])]
        _, want = _check(*args, srh_layer=_layers(500, 23), bwd_layer=_layers(500, 24))
    assert np.isfinite(want["bunkers_right_u"]).mean() > 0.9


def test_read_extent_and_requests():
    """The column is read up to the first profile point at or above the highest bound the call needs, and only the
    requested parts set it."""
    z, u, v, su, sv = _sheared(300, 45, seed=31)
    full = _check(z, u, v, su, sv)[0]
    first = lambda h: np.argmax(np.where(np.isnan(z), -1, z) >= h, axis=0) + 1   # noqa: E731
    assert np.array_equal(full["levels_read"], first(6000.0))
    bwd_only = _check(z, u, v, su, sv, depths=(), bwd_layer=(np.zeros(300), np.full(300, 2000.0)), motion=False)[0]
    assert np.array_equal(bwd_only["levels_read"], first(2000.0))
    assert np.array_equal(bwd_only["bulk_wind_difference"], _check(z, u, v, su, sv, bwd_layer=(
        np.zeros(300), np.full(300, 2000.0)))[0]["bulk_wind_difference"])
    nothing = hs.storm_kinematics(z, u, v, su, sv, 1, (), motion=False)
    assert (nothing["levels_read"] == 0).all()


def _one(z, u, v, su=0.0, sv=0.0, **kw):
    col = lambda x: np.asarray(x, np.float64)[:, None]                      # noqa: E731
    return _check(col(z), col(u), col(v), [su], [sv], **kw)[0]


def test_hand_built_columns():
    z = [100.0, 500.0, 1200.0, 3000.0, 5500.0, 6000.0, 7000.0]
    u = [1.0, 4.0, 8.0, 15.0, 20.0, 22.0, 25.0]
    v = [0.5, 2.0, 1.0, -2.0, -1.0, 3.0, 4.0]
    r = _one(z, u, v, srh_layer=([500.0], [500.0]), bwd_layer=([-50.0], [5500.0]))
    assert np.isfinite(r["bunkers_right_u"][0]) and r["srh_layer"][0] == 0.0
    assert r["bulk_wind_difference_u"][0] == 20.0 and r["bulk_wind_difference_v"][0] == -1.0    # from the surface
    # a profile ending just below 6 km: no motion, no SRH; a BWD below the top still defined
    r = _one(z[:4] + [5999.9], u[:5], v[:5], bwd_layer=([0.0], [3000.0]))
    assert np.isnan(r["bunkers_right_u"][0]) and np.isnan(r["srh_0_1000m"][0])
    assert r["bulk_wind_difference_u"][0] == 15.0
    # non-increasing kept heights below the extent: everything NaN; above it: not read
    r = _one([100.0, 500.0, 500.0, 3000.0, 6000.0], u[:5], v[:5], bwd_layer=([0.0], [1000.0]))
    assert all(np.isnan(r[k][0]) for k in MOTION + BWD)
    r = _one(z + [6500.0], u + [1.0], v + [1.0])
    assert np.isfinite(r["bunkers_right_u"][0]) and r["levels_read"][0] == 6
    # NaN surface wind
    r = _one(z, u, v, su=np.nan, bwd_layer=([0.0], [1000.0]))
    assert all(np.isnan(r[k][0]) for k in MOTION + BWD)
    # reversed layer, negative bound, NaN bound, a bound above the profile
    for lay, finite in ((([2000.0], [1000.0]), False), (([-300.0], [-100.0]), True), (([-300.0], [800.0]), True),
                        (([np.nan], [800.0]), False), (([100.0], [8000.0]), False)):
        r = _one(z, u, v, srh_layer=lay, bwd_layer=lay)
        assert np.isfinite(r["srh_layer"][0]) == finite and np.isfinite(r["bulk_wind_difference"][0]) == finite, lay
    r = _one(z, u, v, srh_layer=([-300.0], [-100.0]), bwd_layer=([-300.0], [-100.0]))
    assert r["srh_layer"][0] == 0.0 and r["bulk_wind_difference"][0] == 0.0                     # [0, 0]
    # levels below ground and with a NaN are dropped
    r2 = _one([-20.0, 0.0] + z[:3] + [np.nan] + z[3:], [50.0, 50.0] + u[:3] + [1.0] + u[3:],
              [50.0, 50.0] + v[:3] + [1.0] + v[3:])
    r1 = _one(z, u, v)
    for k in MOTION + ["srh_0_1000m", "srh_0_3000m"]:
        assert r1[k][0] == r2[k][0], k


# ---- composites -----------------------------------------------------------------------------------------------------
def test_composite_thresholds_exactly():
    ebwd = np.array([9.999, 10.0, 15.0, 20.0, 20.001, 12.4999, 12.5, 30.0, 30.001, np.nan])
    scp, _ = hs.composites(2000.0, 100.0, ebwd, 1500.0, 0.0, 500.0)
    want_tb = np.array([0.0, 0.5, 0.75, 1.0, 1.0, 0.62499500, 0.625, 1.0, 1.0, np.nan])
    assert np.allclose(scp, 2.0 * 2.0 * want_tb, rtol=1e-15, equal_nan=True)
    _, stp = hs.composites(1.0, 150.0, ebwd, 1500.0, 0.0, 500.0)
    tb = np.array([0.0, 0.0, 0.75, 1.0, 1.00005, 0.0, 0.625, 1.5, 1.5, np.nan])
    assert np.allclose(stp, tb, rtol=1e-15, equal_nan=True)
    lcl = np.array([999.0, 1000.0, 1500.0, 2000.0, 2001.0, np.nan])
    _, stp = hs.composites(1.0, 150.0, 40.0, 1500.0, 0.0, lcl)
    assert np.allclose(stp, 1.5 * np.array([1.0, 1.0, 0.5, 0.0, 0.0, np.nan]), rtol=1e-15, equal_nan=True)
    cin = np.array([-49.0, -50.0, -125.0, -200.0, -201.0, np.nan])
    _, stp = hs.composites(1.0, 150.0, 40.0, 1500.0, cin, 500.0)
    assert np.allclose(stp, 1.5 * np.array([1.0, 1.0, 0.5, 0.0, 0.0, np.nan]), rtol=1e-15, equal_nan=True)
    # max(0, .): negative helicity gives 0, NaN stays NaN; NaN in any input gives NaN, even beside a zero factor
    _, stp = hs.composites(1.0, [-150.0, np.nan], 40.0, [1500.0, 1500.0], 0.0, 500.0)
    assert stp[0] == 0.0 and np.isnan(stp[1])
    scp, stp = hs.composites(np.nan, 100.0, 5.0, np.nan, 0.0, 500.0)
    assert np.isnan(scp) and np.isnan(stp)


def test_composites_against_oracle():
    rng = np.random.default_rng(41)
    n = 20000
    x = [rng.uniform(0, 5000, n), rng.uniform(-300, 600, n), rng.uniform(0, 40, n), rng.uniform(0, 4000, n),
         rng.uniform(-300, 0, n), rng.uniform(0, 3000, n)]
    for a in x:
        a[rng.random(n) < 0.02] = np.nan
    x[2][::97] = np.array([10.0, 20.0, 12.5, 30.0])[np.arange(x[2][::97].size) % 4]
    x[5][::89] = np.array([1000.0, 2000.0])[np.arange(x[5][::89].size) % 2]
    x[4][::83] = np.array([-50.0, -200.0])[np.arange(x[4][::83].size) % 2]
    scp, stp = hs.composites(*x)
    want_scp = ko.supercell_composite(x[0], x[1], x[2])
    want_stp = ko.significant_tornado(x[3], x[1], x[2], x[5], x[4])
    assert np.array_equal(scp, want_scp, equal_nan=True)
    assert np.array_equal(stp, want_stp, equal_nan=True)
