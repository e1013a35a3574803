"""Seeded columns of the real-world regimes that ``xarray_parcel_b200.synth`` does not reach.

synth draws surface pressure from 950-1030 hPa, surface temperature from 270-308 K, a stratosphere of 195-225 K and a
model top at 20 hPa.  Users' grids go further: high terrain (the Tibetan plateau at 550-600 hPa, Antarctica at 600-700
hPa and 220-250 K), moist heat with surface dewpoints near 308 K, model tops at 0.01 hPa (IFS L137, ERA5 model levels),
sea-level extrapolations above 1100 hPa and ERA5 pressure-level data with the below-ground levels masked to NaN.  Those
inputs take other routes through the fast kernels -- the table rows outside segment A, every column handed over to the
float64 fix-up -- and through the downdraft and effective-layer kernels, so the GPU tests draw them from here.

Every regime gives float32 level-major ``[L, N]`` temperature and dewpoint.  ``layout="model"`` puts them on per-column
hybrid-sigma pressure ``[L, N]``; ``"era5"`` on the 37 shared ERA5 levels with the below-ground levels extrapolated
(6.5 K/km, constant dewpoint depression) as ERA5 does; ``"era5_masked"`` the same with the below-ground levels NaN;
``"axis"`` on a deep shared axis of ``levels`` levels up to ``p_top``, extrapolated below ground.
"""

import numpy as np

ERA5_LEVELS_HPA = np.array([1000, 975, 950, 925, 900, 875, 850, 825, 800, 775, 750, 700, 650, 600, 550, 500, 450,
                            400, 350, 300, 250, 225, 200, 175, 150, 125, 100, 70, 50, 30, 20, 10, 7, 5, 3, 2, 1],
                           dtype=np.float64)

# surface pressure (hPa), surface temperature (K), surface dewpoint depression (K), stratosphere temperature (K)
REGIMES = {
    # high terrain: the surface is colder the higher it lies (2 K per km of surface height)
    "terrain": dict(p0=(550.0, 1050.0), t0=(265.0, 305.0), dd=(0.5, 20.0), strat=(195.0, 225.0), terrain=True),
    # polar and plateau cold: Antarctica, Greenland, the winter plateau
    "cold": dict(p0=(600.0, 1040.0), t0=(215.0, 262.0), dd=(0.5, 8.0), strat=(180.0, 215.0)),
    # tropical moist heat: surface dewpoints up to 308 K, a cold tropopause
    "moist_heat": dict(p0=(995.0, 1015.0), t0=(300.0, 315.0), dd=(0.3, 6.0), strat=(185.0, 200.0)),
    # sea-level extrapolation below high ground and deep lows of the reanalysis: 15 % of the columns above 1100 hPa
    "high_surface": dict(p0=(1030.0, 1099.0), t0=(240.0, 300.0), dd=(0.5, 15.0), strat=(195.0, 225.0),
                         above_1100=0.15),
    # only the part above 1100 hPa, where the table of the fast kernels ends
    "above_1100": dict(p0=(1100.5, 1150.0), t0=(240.0, 300.0), dd=(0.5, 15.0), strat=(195.0, 225.0)),
    # the synth ranges, for the deep-top and long-column axes
    "synth_like": dict(p0=(950.0, 1030.0), t0=(270.0, 305.0), dd=(0.5, 15.0), strat=(195.0, 225.0)),
    # the synth thermodynamics over land up to the high plateaus: with layout="era5_masked", ERA5 pressure-level data
    "masked": dict(p0=(550.0, 1030.0), t0=(270.0, 305.0), dd=(0.5, 15.0), strat=(195.0, 225.0), terrain=True),
}

MAX_DEWPOINT = 308.0       # the highest surface dewpoints observed (Persian Gulf, Red Sea)


def _surface_pressure(spec, n, rng):
    p0 = rng.uniform(*spec["p0"], n)
    frac = spec.get("above_1100", 0.0)
    if frac:
        hi = rng.random(n) < frac
        p0[hi] = rng.uniform(1100.5, 1150.0, hi.sum())
    return p0


def _thermo(p, p0, spec, rng):
    """Temperature and dewpoint [L, N] (float64) on pressures ``p`` [L, N] for surface pressures ``p0`` [N]."""
    n = p0.size
    z = 7.5 * np.log(p0[None, :] / p)                               # km above the surface (< 0 below ground)
    t0 = rng.uniform(*spec["t0"], n)
    if spec.get("terrain"):
        t0 = t0 - 2.0 * 7.5 * np.log(1013.25 / p0)
    lapse = rng.uniform(5.0, 9.5, n)
    t_strat = rng.uniform(*spec["strat"], n)
    above = np.maximum(t0[None, :] - lapse[None, :] * z, t_strat[None, :])
    t = np.where(z >= 0, above, t0[None, :] - 6.5 * z)               # below ground: ERA5's extrapolation
    dd = rng.uniform(*spec["dd"], n)[None, :] + 1.5 * np.clip(z, 0.0, 15.0)
    td = np.minimum(t - dd, MAX_DEWPOINT)
    return t, td


def _model_pressure(p0, levels, p_top):
    s = np.arange(levels, dtype=np.float64) / (levels - 1)
    if p_top >= 20.0:
        sigma = 1.0 - s ** 1.6                                       # as synth: finer spacing near the surface
        return p_top + (p0[None, :] - p_top) * sigma[:, None]
    # a deep top (IFS L137-like): even in ln p aloft, fine near the surface
    sigma = 1.0 - s ** 1.3
    return np.exp(np.log(p0)[None, :] * sigma[:, None] + np.log(p_top) * (1.0 - sigma[:, None]))


def axis_pressure(regime, levels, p_top):
    """The shared axis of ``layout="axis"``: ``levels`` pressures [hPa] spaced as the hybrid-sigma levels of a column
    whose surface is the regime's highest surface pressure (1150 hPa where columns lie above 1100 hPa)."""
    spec = REGIMES[regime]
    p_bottom = 1150.0 if spec.get("above_1100") else spec["p0"][1]
    return _model_pressure(np.array([p_bottom]), levels, p_top)[:, 0]


def columns(regime, n, seed, layout="model", levels=70, p_top=20.0):
    """(p, T, Td, p0) of ``n`` columns of ``regime``: float32 arrays (p [L, N] for ``layout="model"``, [37] for the
    ERA5 layouts, [levels] for ``layout="axis"``) and the float64 surface pressure [N] the columns were drawn for.
    ``"axis"`` is a deep shared axis (``axis_pressure``) with the below-ground levels extrapolated as in ``"era5"``."""
    spec = REGIMES[regime]
    rng = np.random.default_rng(seed)
    p0 = _surface_pressure(spec, n, rng)
    if layout == "model":
        p32 = _model_pressure(p0, levels, p_top).astype(np.float32)
        assert (np.diff(p32, axis=0) < 0).all(), "pressure must decrease strictly with level"
        t, td = _thermo(p32.astype(np.float64), p0, spec, rng)
    elif layout == "axis":
        p32 = axis_pressure(regime, levels, p_top).astype(np.float32)
        assert (np.diff(p32) < 0).all(), "pressure must decrease strictly with level"
        t, td = _thermo(np.broadcast_to(p32.astype(np.float64)[:, None], (levels, n)), p0, spec, rng)
    else:
        assert layout in ("era5", "era5_masked"), layout
        p32 = ERA5_LEVELS_HPA.astype(np.float32)
        t, td = _thermo(np.broadcast_to(ERA5_LEVELS_HPA[:, None], (37, n)), p0, spec, rng)
    t32 = t.astype(np.float32)
    td32 = np.minimum(td.astype(np.float32), t32)
    if layout == "era5_masked":
        below = ERA5_LEVELS_HPA[:, None] > p0[None, :]
        t32[below] = np.nan
        td32[below] = np.nan
    return p32, np.ascontiguousarray(t32), np.ascontiguousarray(td32), p0


def conv_fields(p, t, td, p0, seed, dry_top_every=53, negative_q_every=211):
    """The ``conv_properties`` input dict of a regime's columns ``(p, T, Td, p0)``, float32 throughout.

    specific_humidity from Td (NaN where Td is masked).  height_asl is hypsometric on the float64 virtual temperature
    from a surface at 7.5 km * ln(1013.25 / p0) and stays finite on extrapolated and masked levels, as ERA5 geopotential
    does (a masked level takes the virtual temperature of the lowest valid level).  Winds are seeded sheared profiles,
    NaN where T is masked; wind_height_above_surface = height_asl - surface height, negative below ground;
    surface_wind_u / _v are per-column.  Every ``dry_top_every``-th column (from column 3) has q exactly 0 on its top two
    levels and every ``negative_q_every``-th (from column 7) -1e-7 there, as model output can carry both."""
    rng = np.random.default_rng(seed)
    L, n = t.shape
    q = specific_humidity(p, td)
    # a warm layer (up to +8 K, 800 m deep, 0.3-3 km above the surface) in every fourth column: inversions that cross
    # 0 C several times where the column is near freezing there
    P = np.broadcast_to(np.asarray(p, np.float64).reshape(L, -1), (L, n))
    z = 7.5 * np.log(p0[None, :] / P)
    bump = rng.uniform(2.0, 8.0, n) * (np.arange(n) % 4 == 1)
    t = (t + bump[None, :] * np.clip(1.0 - np.abs(z - rng.uniform(0.3, 3.0, n)[None, :]) / 0.4, 0.0, None)).astype(
        np.float32)
    q[-2:, 3::dry_top_every] = 0.0
    q[-2:, 7::negative_q_every] = -1e-7
    T = t.astype(np.float64)
    Q = np.nan_to_num(q.astype(np.float64), nan=0.0)
    tv = T * (1.0 + 0.608 * Q / (1.0 - Q))
    valid = ~np.isnan(tv)
    first = np.argmax(valid, axis=0)                                   # lowest valid level (0 if none)
    lowest = np.where(valid.any(axis=0), tv[first, np.arange(n)], 250.0)
    for k in range(L - 1, -1, -1):                                     # masked levels: the lowest valid Tv below
        tv[k] = np.where(np.isnan(tv[k]), lowest, tv[k])
    rd_g = 287.04749097718457 / 9.80665
    z_sfc = 7500.0 * np.log(1013.25 / p0)
    h = np.empty((L, n))
    h[0] = z_sfc + rd_g * tv[0] * np.log(p0 / P[0])                   # negative offset when level 0 is below ground
    for k in range(1, L):
        h[k] = h[k - 1] + rd_g * 0.5 * (tv[k - 1] + tv[k]) * np.log(P[k - 1] / P[k])
    agl = h - z_sfc[None, :]
    km = np.clip(agl, 0.0, None) / 1000.0
    u = rng.normal(3.0, 5.0, n)[None, :] + rng.uniform(-1.0, 6.0, n)[None, :] * km + rng.normal(0.0, 1.5, (L, n))
    v = rng.normal(0.0, 5.0, n)[None, :] + rng.uniform(-3.0, 3.0, n)[None, :] * km + rng.normal(0.0, 1.5, (L, n))
    masked = np.isnan(t)
    u[masked] = np.nan
    v[masked] = np.nan
    f32 = lambda x: np.ascontiguousarray(x, dtype=np.float32)                  # noqa: E731
    return {"pressure": np.asarray(p, np.float32), "temperature": f32(t), "specific_humidity": f32(q),
            "height_asl": f32(h), "wind_u": f32(u), "wind_v": f32(v), "wind_height_above_surface": f32(agl),
            "surface_wind_u": f32(rng.normal(2.0, 4.0, n)), "surface_wind_v": f32(rng.normal(0.0, 4.0, n))}


def specific_humidity(p, td):
    """float32 specific humidity [kg/kg] of dewpoint ``td`` [K] at ``p`` [hPa] (Bolton's vapour pressure)."""
    p = np.asarray(p, np.float64)
    if p.ndim == 1:
        p = p[:, None]
    tc = np.asarray(td, np.float64) - 273.15
    e = 6.112 * np.exp(17.67 * tc / (tc + 243.5))
    w = 0.622 * e / (p - e)
    return (w / (1.0 + w)).astype(np.float32)
