"""Downdraft CAPE: the column code of xp_downdraft.cuh (host-compiled from tests/hostsim/hostsim_downdraft.cpp)
against the NumPy restatement of the contract (tests/downdraft_oracle.py, DESIGN.md section 3.12), on synthetic,
lattice and hand-built columns."""

import numpy as np
import pytest

import downdraft_oracle as dd
import hostsim_downdraft as hs
from oracle import parcel as op
from oracle import thermo as th
from test_lattice_soundings import lattice_columns
from xarray_parcel_b200 import synth

COMPAT = {"1.4.1": 141, "1.6.2": 162}


@pytest.fixture(scope="module")
def lut(oracle_tables):
    return op.Options(op.MoistLapseLUT(oracle_tables), lcl_mode="converged")


def _opts(tables, compat):
    return op.Options(op.MoistLapseLUT(tables), metpy_compat=compat, lcl_mode="converged")


def _check(P, T, D, tables, compat="1.4.1"):
    ora = dd.downdraft_cape(P, T, D, _opts(tables, compat))
    got = hs.downdraft_cape(P, T, D, tables, metpy_compat=COMPAT[compat], profile=True)
    p2 = np.broadcast_to(op._as2d(P), T.shape)
    dd.assert_matches(got, ora, op.nanmax(np.where(np.isnan(T) | np.isnan(D), np.nan, p2)),
                      ora["downdraft_start_pressure"])
    return got, ora


def _one(tables, p, t, td, compat="1.4.1"):
    """One hand-built column through both; returns the host result (scalars as floats)."""
    P, T, D = [np.asarray(x, dtype=np.float64)[:, None] for x in (p, t, td)]
    got, ora = _check(P, T, D, tables, compat)
    return {k: (v[0] if v.ndim == 1 else v[:, 0]) for k, v in got.items()}


@pytest.mark.parametrize("compat", ["1.4.1", "1.6.2"])
@pytest.mark.parametrize("shape", ["model70", "era5"])
def test_synthetic_columns_match_oracle(oracle_tables, shape, compat):
    """NaN levels, all-NaN columns and a fifth of the columns saturated at the surface."""
    if shape == "model70":
        p, t, td = synth.model_level_columns(4000, 70, seed=21, nan_columns=0.05, allnan_columns=0.01, saturated=0.2)
    else:
        p, t, td = synth.era5_columns(4000, seed=22, nan_columns=0.05, allnan_columns=0.01, saturated=0.2)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    got, ora = _check(P, T, D, oracle_tables, compat)
    assert np.isnan(ora["dcape"]).mean() < 0.05                     # the all-NaN columns and little else
    assert (ora["dcape"] > 0).mean() > 0.8


def test_fully_saturated_columns_match_oracle(oracle_tables):
    p, t, _ = synth.model_level_columns(1500, 70, seed=23, nan_columns=0.0, allnan_columns=0.0)
    P, T = [x.numpy().astype(np.float64) for x in (p, t)]
    _check(P, T, T.copy(), oracle_tables)


def test_era5_reads_no_level_beyond_the_first_valid_level_past_500_hpa(oracle_tables):
    """On the ERA5 axis that is the 450 hPa level: 17 of the 37 levels (a level within np.isclose below 500 hPa would
    still be a candidate, so the first level past it has to be read)."""
    p, t, td = synth.era5_columns(500, seed=24)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    got = hs.downdraft_cape(P, T, D, oracle_tables)
    assert got["levels_read"].max() == synth.ERA5_LEVELS_HPA.index(450) + 1 == 17


@pytest.mark.parametrize("compat", ["1.4.1", "1.6.2"])
@pytest.mark.parametrize("L,dp", [(20, 25.0), (24, 20.0), (10, 50.0), (16, 50.0)])
def test_lattice_soundings_match_oracle(oracle_tables, L, dp, compat):
    """Pressures on a 20-50 hPa lattice land exactly on 700 and 500 hPa in most columns; a quarter of those levels
    are moved to within (or just outside) np.isclose of the bound."""
    n = 1500
    p, t, td = lattice_columns(n, L, 300 + L, dp)
    r = np.random.default_rng(L)
    for bound in (700.0, 500.0):
        on = (p == bound) & (r.random(p.shape) < 0.25)
        jitter = r.choice([-0.0069, 0.0069, -0.0071, 0.0071, 0.003], size=p.shape)
        p = np.where(on, bound + jitter, p)
    ora = dd.downdraft_cape(p, t, td, _opts(oracle_tables, compat))
    got = hs.downdraft_cape(p, t, td, oracle_tables, metpy_compat=COMPAT[compat], profile=True)
    pmax = op.nanmax(np.where(np.isnan(t) | np.isnan(td), np.nan, p))
    dd.assert_matches(got, ora, pmax, ora["downdraft_start_pressure"])
    assert (~np.isnan(ora["dcape"])).sum() > 0.3 * n


# ---- contract cases ------------------------------------------------------------------------------------------------
P8 = [1000.0, 925.0, 850.0, 700.0, 600.0, 500.0, 400.0, 300.0]
T8 = [300.0, 295.0, 290.0, 280.0, 272.0, 262.0, 250.0, 235.0]
D8 = [292.0, 288.0, 282.0, 262.0, 255.0, 245.0, 230.0, 215.0]


def test_surface_below_700_hpa_gives_nan(oracle_tables):
    r = _one(oracle_tables, [690.0] + P8[4:], [281.0] + T8[4:], [263.0] + D8[4:])
    assert np.isnan(r["dcape"]) and np.isnan(r["downdraft_start_pressure"]) and np.isnan(r["downdraft_start_temperature"])
    assert np.isnan(r["downdraft_parcel_temperature"]).all()


def test_top_above_500_hpa_gives_nan(oracle_tables):
    r = _one(oracle_tables, P8[:5] + [510.0], T8[:5] + [263.0], D8[:5] + [246.0])
    assert np.isnan(r["dcape"]) and np.isnan(r["downdraft_start_pressure"])


def test_a_level_within_isclose_of_700_is_used_instead_of_an_interpolated_point(oracle_tables):
    """The driest level sits next to 700 hPa: within np.isclose (0.007 hPa) it is the start itself; just outside,
    the start is the point interpolated at exactly 700 hPa."""
    t = [300.0, 295.0, 290.0, 280.0, 272.0, 262.0, 250.0, 235.0]
    d = [292.0, 288.0, 282.0, 240.0, 262.0, 250.0, 230.0, 215.0]
    for p700, start in ((700.006, 700.006), (699.994, 699.994), (700.0071, 700.0), (699.9929, 700.0)):
        p = list(P8)
        p[3] = p700
        r = _one(oracle_tables, p, t, d)
        assert r["downdraft_start_pressure"] == start, p700
        assert np.isfinite(r["dcape"])


def test_one_descent_level_gives_zero(oracle_tables):
    """The surface at 700 hPa is the start: the descent is that one level and the integral is 0."""
    r = _one(oracle_tables, P8[3:], [280.0, 275.0, 270.0, 255.0, 240.0], [240.0, 262.0, 255.0, 230.0, 215.0])
    assert r["downdraft_start_pressure"] == 700.0
    assert r["dcape"] == 0.0
    assert np.isfinite(r["downdraft_parcel_temperature"][0]) and np.isnan(r["downdraft_parcel_temperature"][1:]).all()


def test_a_nan_level_is_the_same_as_the_level_removed(oracle_tables):
    for drop in (1, 3, 4, 5):
        t_nan = list(T8)
        t_nan[drop] = np.nan
        a = _one(oracle_tables, P8, t_nan, D8)
        b = _one(oracle_tables, P8[:drop] + P8[drop + 1:], T8[:drop] + T8[drop + 1:], D8[:drop] + D8[drop + 1:])
        for k in ("dcape", "downdraft_start_pressure", "downdraft_start_temperature"):
            assert a[k] == b[k], (drop, k)
        assert np.isnan(a["downdraft_parcel_temperature"][drop])
        keep = np.delete(a["downdraft_parcel_temperature"], drop)
        assert np.array_equal(keep, b["downdraft_parcel_temperature"], equal_nan=True)


def test_saturated_environment_on_one_adiabat_is_within_one_adiabat_step(oracle_tables):
    """T = Td = one table adiabat at every level.  Two lookups stand between the environment and the descent: the
    wet bulb (the adiabat of the LCL's cell, here the start itself) and the descent adiabat (the cell of the start
    and the wet bulb).  Each picks an adiabat that passes through the nearest 0.02 K cell, so at most 0.03 K off
    (half a cell to the node, one cell width); the parcel starts within 0.06 K of the environment's adiabat and
    below the start the two curves spread as the table's adiabats do (0.03-0.05 K seen at the start here).
    Bound: Rd * 1.5 * step * ln(p_sfc / p_start), step = the largest difference over the descent between the
    environment's adiabat and the adiabats 0.06 K warmer / colder at the start (1.5: the virtual-temperature factor
    of the saturated parcel)."""
    tb = oracle_tables
    xp = tb.pressure_asc
    curves = tb.curves_asc.astype(np.float64)
    p = np.array([1000.0, 950.0, 900.0, 850.0, 800.0, 750.0, 700.0, 650.0, 600.0, 550.0, 500.0, 450.0])
    for j in (6000, 7500, 9000):
        t = np.interp(p, xp, curves[j - 1])
        r = _one(tb, p, t, t.copy())
        ps = r["downdraft_start_pressure"]
        at_ps = curves[:, np.searchsorted(xp, ps)]
        env_ps = np.interp(ps, xp, curves[j - 1])
        desc = p >= ps
        step = 0.0
        for off in (-0.06, 0.06):
            k = np.nanargmin(np.abs(at_ps - (env_ps + off)))
            step = max(step, np.abs(np.interp(p[desc], xp, curves[k]) - t[desc]).max())
        bound = th.RD * 1.5 * step * np.log(p[0] / ps)
        assert np.isfinite(r["dcape"]) and abs(r["dcape"]) < bound, (j, r["dcape"], bound)


def test_a_parcel_warmer_than_the_environment_gives_negative_dcape(oracle_tables):
    """A deep cold pool under moist mid levels: the descending parcel is warmer than the air below it."""
    p = [1000.0, 950.0, 900.0, 850.0, 800.0, 700.0, 600.0, 500.0, 400.0]
    t = [262.0, 262.5, 263.0, 263.0, 262.5, 261.0, 256.0, 248.0, 238.0]
    d = [260.0, 260.5, 261.0, 261.0, 260.5, 259.0, 254.0, 246.0, 230.0]
    r = _one(oracle_tables, p, t, d)
    assert r["dcape"] < -10.0


def test_lut_oracle_agrees_with_the_ode_oracle_on_the_reference_soundings(soundings, oracle_tables):
    """The table's published error carried through the integral: |dcape(LUT) - dcape(ODE)| <= Rd * 0.06 K *
    ln(p_sfc / p_start) * 1.5, where 0.06 K = the 0.037 K table error (in the wet bulb and along the descent) + one
    0.02 K cell at the descent lookup, and 1.5 is the virtual-temperature factor of the saturated parcel."""
    names = [n for n, s in soundings.items() if {"levels", "temperatures", "dewpoints"} <= set(s)
             and np.nanmax(s["levels"]) >= 700.0 and np.nanmin(s["levels"]) <= 500.0]
    assert len(names) >= 5
    for n in names:
        s = soundings[n]
        P, T, D = [s[k][:, None] for k in ("levels", "temperatures", "dewpoints")]
        a = dd.downdraft_cape(P, T, D, op.Options(op.MoistLapseLUT(oracle_tables)))
        b = dd.downdraft_cape(P, T, D, op.Options(op.MoistLapseODE()))
        assert a["downdraft_start_pressure"][0] == b["downdraft_start_pressure"][0], n
        bound = th.RD * 0.06 * np.log(np.nanmax(P) / a["downdraft_start_pressure"][0]) * 1.5
        assert abs(a["dcape"][0] - b["dcape"][0]) <= bound, (n, a["dcape"][0], b["dcape"][0], bound)


def test_conv_properties_oracle_adds_dcape_only_on_request(lut):
    p, t, td = synth.model_level_columns(40, 40, seed=25, nan_columns=0.1, allnan_columns=0.0)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    q = th.saturation_mixing_ratio(P, D)
    q = q / (1 + q)
    H = 7500.0 * np.log(P[0][None, :] / P)
    dat = {"pressure": P, "temperature": T, "specific_humidity": q, "height_asl": H, "wind_u": H / 1000,
           "wind_v": -H / 2000, "wind_height_above_surface": H, "surface_wind_u": np.zeros(40),
           "surface_wind_v": np.zeros(40)}
    base = dd.conv_properties(dat, lut)
    with_dd = dd.conv_properties(dat, lut, downdraft=True)
    assert "dcape" not in base and set(with_dd) == set(base) | {"dcape"}
    td = th.dewpoint_from_specific_humidity(P, T, q)
    expect = dd.downdraft_cape(P, T, td, lut)["dcape"]
    masked = np.isnan(base["mixed_100_cape"])
    assert np.isnan(with_dd["dcape"][masked]).all()
    assert np.array_equal(with_dd["dcape"][~masked], expect[~masked], equal_nan=True)
