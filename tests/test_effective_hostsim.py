"""Effective inflow layer: the column code of xp_effective.cuh (host-compiled from tests/hostsim/hostsim_effective.cpp)
against the NumPy restatement of the contract (tests/effective_oracle.py, DESIGN.md section 3.13), on synthetic,
lattice and hand-built columns, in search mode and in all-levels mode."""

import numpy as np
import pytest

import effective_oracle as eo
import hostsim_effective as hs
from oracle import parcel as op
from test_lattice_soundings import lattice_columns
from xarray_parcel_b200 import synth

OPTIONS = [dict(metpy_compat="1.4.1"),
           dict(metpy_compat="1.6.2", virtual_temperature_correction=False),
           dict(metpy_compat="1.4.1", pos_cape_neg_cin=False),
           dict(metpy_compat="1.6.2", virtual_temperature_correction=False, pos_cape_neg_cin=False)]
OPTION_IDS = ["defaults", "1.6.2-no-vtc", "no-pos-neg", "1.6.2-no-vtc-no-pos-neg"]


def _run(P, T, D, tables, opt=None, min_cape=100.0, min_cin=-250.0, depth=300.0):
    """Both through the oracle and the host build; checks everything the contract pins and returns (host, oracle,
    excused level count)."""
    opt = dict(opt or {})
    compat = opt.pop("metpy_compat", "1.4.1")
    opts = op.Options(op.MoistLapseLUT(tables), metpy_compat=compat, lcl_mode="converged")
    ora = eo.effective_inflow_layer(P, T, D, opts, min_cape, min_cin, depth, **opt)
    got = hs.effective_inflow_layer(P, T, D, tables, min_cape, min_cin, depth,
                                    metpy_compat=141 if compat == "1.4.1" else 162, **opt)
    p2 = np.broadcast_to(op._as2d(P), T.shape)
    valid = eo.valid_levels(P, T, D)
    # per-level CAPE / CIN at 1e-9 relative (1 J/kg floor), identical NaN patterns; saturated starts excused
    excuse = valid & (T == D)
    for a, b in (("level_cape", "level_parcel_cape"), ("level_cin", "level_parcel_cin")):
        x, y = got[a], ora[b]
        assert np.array_equal(np.isnan(x), np.isnan(y)), a
        assert np.array_equal(np.isnan(x), ~valid), a
        with np.errstate(invalid="ignore"):
            err = np.where(np.isnan(y), 0.0, np.abs(x - y) / np.maximum(np.abs(y), 1.0))
        assert not (err[~excuse] > 1e-9).any(), (a, np.nanmax(err[~excuse]))
    # the search, bit for bit: on the column code's own per-level values, and both modes alike
    base_k, top_k = eo.search(got["level_cape"], got["level_cin"], got["gate"], valid, min_cape, min_cin)
    for k, lv in (("base", base_k), ("top", top_k)):
        want = eo.level_pressure(P, T.shape, lv)
        assert np.array_equal(got[k], want, equal_nan=True), k
        assert np.array_equal(got["all_" + k], want, equal_nan=True), "all_" + k
    # base / top against the oracle's, excusing columns with a value within 1e-6 J/kg of a threshold or a saturated
    # level (where the level values may differ)
    with np.errstate(invalid="ignore"):
        near = (np.abs(ora["level_parcel_cape"] - min_cape) < 1e-6) | (np.abs(ora["level_parcel_cin"] - min_cin) < 1e-6)
    loose = (near | excuse).any(axis=0)
    for k in ("base", "top"):
        same = np.isclose(got[k], ora["effective_inflow_" + k], rtol=0, atol=0, equal_nan=True)
        assert (same | loose).all(), (k, np.flatnonzero(~(same | loose))[:5])
    assert got["flags"] == (0, 0)
    assert np.array_equal(got["gate"] | loose, ora["gate"] | loose)
    return got, ora, int(excuse.sum()), p2


@pytest.mark.parametrize("opt", OPTIONS, ids=OPTION_IDS)
@pytest.mark.parametrize("shape", ["era5", "model70"])
def test_synthetic_columns_match_oracle(oracle_tables, shape, opt):
    if shape == "era5":
        p, t, td = synth.era5_columns(600, seed=41, nan_columns=0.05, allnan_columns=0.01)
    else:
        p, t, td = synth.model_level_columns(250, 70, seed=42, nan_columns=0.05, allnan_columns=0.01)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    got, ora, excused, _ = _run(P, T, D, oracle_tables, opt)
    assert excused <= 0.01 * T.size
    have = ~np.isnan(ora["effective_inflow_base"])
    assert 0.2 < have.mean() < 0.8                                   # both outcomes well represented
    assert (ora["effective_inflow_base"][have] >= ora["effective_inflow_top"][have]).all()


@pytest.mark.parametrize("opt", OPTIONS[:2], ids=OPTION_IDS[:2])
@pytest.mark.parametrize("L,dp", [(20, 25.0), (12, 40.0), (4, 50.0), (2, 25.0), (1, 25.0)])
def test_lattice_columns_match_oracle(oracle_tables, L, dp, opt):
    """Lattice pressures with NaN T / Td levels, trailing NaN pressures and T == Td levels."""
    p, t, td = lattice_columns(800, L, 500 + L, dp)
    _, _, excused, _ = _run(p, t, td, oracle_tables, opt)
    assert excused <= 0.1 * t.size


def test_seed_1234_gate_fails_although_a_lower_level_passes(oracle_tables):
    """The rare case (about 0.4 % of the seed-1234 ERA5 columns): the most-unstable parcel fails, a lower level
    passes, and the column has no layer."""
    p, t, td = synth.era5_columns(1500, seed=1234)
    P, T, D = [x.numpy().astype(np.float64) for x in (p, t, td)]
    got, ora, _, _ = _run(P, T, D, oracle_tables)
    any_pass = (eo.passes(ora["level_parcel_cape"], ora["level_parcel_cin"])).any(axis=0)
    case = ~ora["gate"] & any_pass
    assert case.sum() >= 1
    assert np.isnan(got["base"][case]).all() and np.isnan(got["all_base"][case]).all()
    # the surface is not always the base: elevated bases occur
    have = ~np.isnan(got["base"])
    assert (got["base"][have] < P[0]).any()


# ---- hand-built columns --------------------------------------------------------------------------------------------
P10 = [1000.0, 950.0, 900.0, 850.0, 800.0, 700.0, 600.0, 500.0, 400.0, 300.0]
T10 = [303.0, 299.0, 296.0, 293.0, 290.0, 283.0, 275.0, 265.0, 252.0, 236.0]
D10 = [297.0, 294.0, 291.0, 288.0, 282.0, 270.0, 255.0, 240.0, 225.0, 210.0]


def _one(tables, p, t, td, **kw):
    P, T, D = [np.asarray(x, dtype=np.float64)[:, None] for x in (p, t, td)]
    got, ora, _, _ = _run(P, T, D, tables, **kw)
    return {k: (v[0] if v.ndim == 1 else v[:, 0]) for k, v in got.items() if k != "flags"}, ora


def test_moist_column_has_a_surface_based_layer(oracle_tables):
    r, _ = _one(oracle_tables, P10, T10, D10)
    assert r["base"] == 1000.0 and np.isfinite(r["top"]) and r["top"] < r["base"]
    assert (r["level_cape"][P10.index(r["base"])] >= 100.0)


def test_stable_surface_layer_under_an_elevated_base(oracle_tables):
    """A cold, dry surface layer: its parcels fail; the base is above it."""
    t = [285.0, 287.0, 296.0] + T10[3:]
    d = [270.0, 272.0, 291.0] + D10[3:]
    r, _ = _one(oracle_tables, P10, t, d)
    assert r["base"] == 900.0 and r["top"] <= 900.0
    assert not eo.passes(r["level_cape"][:2], r["level_cin"][:2]).any()


def test_one_level_layer(oracle_tables):
    """Thresholds set between the CAPE of the base parcel and that of the parcel above it."""
    r, _ = _one(oracle_tables, P10, T10, D10, min_cape=0.0, min_cin=-1e9)
    cape = r["level_cape"]
    thr = 0.5 * (cape[0] + cape[1]) if cape[0] > cape[1] else None
    assert thr is not None
    r2, _ = _one(oracle_tables, P10, T10, D10, min_cape=thr, min_cin=-1e9)
    assert r2["base"] == r2["top"] == 1000.0


def test_nan_levels_inside_the_layer_are_skipped(oracle_tables):
    """A NaN temperature inside the layer: that level is neither lifted nor the top; the top skips back to the last
    valid level below the first failing one."""
    r, _ = _one(oracle_tables, P10, T10, D10)
    k_top = P10.index(r["top"])
    assert k_top >= 1
    t = list(T10)
    t[k_top] = np.nan
    r2, _ = _one(oracle_tables, P10, t, D10)
    assert np.isnan(r2["level_cape"][k_top])
    assert r2["top"] != P10[k_top]


def test_non_default_thresholds(oracle_tables):
    a, _ = _one(oracle_tables, P10, T10, D10)
    b, _ = _one(oracle_tables, P10, T10, D10, min_cape=1e6)            # nothing passes
    assert np.isnan(b["base"]) and np.isnan(b["top"])
    c, _ = _one(oracle_tables, P10, T10, D10, min_cape=0.0, min_cin=-1e9)   # the gate and most levels pass
    assert c["base"] == 1000.0
    assert np.array_equal(a["level_cape"], c["level_cape"], equal_nan=True)


def test_degenerate_columns(oracle_tables):
    nan = np.nan
    # one valid level, an all-NaN column, trailing NaN pressures, a NaN surface level
    p = np.array([[1000.0, nan, 1000.0, 1000.0], [900.0, nan, 900.0, 900.0], [800.0, nan, nan, 800.0]])
    t = np.array([[nan, nan, 300.0, 301.0], [296.0, nan, 295.0, 296.0], [290.0, nan, nan, 290.0]])
    d = np.array([[nan, nan, 296.0, 297.0], [294.0, nan, 292.0, 293.0], [288.0, nan, nan, 287.0]])
    for mc in (100.0, 0.0):
        got, ora, _, _ = _run(p, t, d, oracle_tables, min_cape=mc, min_cin=-1e9)
        assert np.isnan(got["level_cape"][:, 1]).all() and np.isnan(got["base"][1])
        assert np.isnan(got["level_cape"][2, 2]) and np.isnan(got["level_cape"][0, 0])
    # a column of one level
    got, _, _, _ = _run(np.array([[1000.0]]), np.array([[300.0]]), np.array([[295.0]]), oracle_tables)
    assert got["level_cape"][0, 0] == 0.0 and np.isnan(got["base"][0])
