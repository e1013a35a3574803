"""NumPy float64 restatement of downdraft CAPE (DESIGN.md section 3.12), the reference the DCAPE kernel is tested
against.  It follows MetPy's ``downdraft_cape`` recipe step for step on the oracle's thermodynamics and its pluggable
moist adiabat (``oracle.parcel.MoistLapseLUT`` / ``MoistLapseODE``), the way ``oracle.parcel.wet_bulb_temperature``
and ``parcel_profile`` do.  It lives beside the tests and leaves the ``oracle`` package, which the other tests pin,
unchanged.

Arrays are level-major ``[L, N]`` (level 0 = surface, pressure decreasing with the level index); pressure may be a
shared ``[L]`` axis."""

import numpy as np

from oracle import parcel as op
from oracle import thermo as th

BOTTOM, TOP = 700.0, 500.0


def _close(p, bound):
    """np.isclose(p, bound)."""
    return abs(p - bound) <= 1e-8 + 1e-5 * bound


def _interp(vb, va, pb, pa, x):
    """Linear in ln p between the bracketing valid levels; b is the one of larger pressure."""
    return vb + (np.log(x) - np.log(pb)) * (va - vb) / (np.log(pa) - np.log(pb))


def _start(p, t, td):
    """Steps 1-3 for one column: (p_s, T_s, Td_s, descent level indices) or None (every output NaN)."""
    valid = np.flatnonzero(~(np.isnan(p) | np.isnan(t) | np.isnan(td)))
    if valid.size < 2:
        return None
    pv, tv, dv = p[valid], t[valid], td[valid]
    c700 = np.array([_close(x, BOTTOM) for x in pv])
    c500 = np.array([_close(x, TOP) for x in pv])
    if (pv.max() < BOTTOM and not c700.any()) or (pv.min() > TOP and not c500.any()):
        return None
    cand = [(x, a, b) for x, a, b, k7, k5 in zip(pv, tv, dv, c700, c500)
            if (x <= BOTTOM or k7) and (x >= TOP or k5)]
    for bound, close in ((BOTTOM, c700), (TOP, c500)):
        if not close.any():
            ib = np.flatnonzero(pv > bound)[-1]                       # the bracketing valid levels
            ia = np.flatnonzero(pv < bound)[0]
            cand.append((bound, _interp(tv[ib], tv[ia], pv[ib], pv[ia], bound),
                         _interp(dv[ib], dv[ia], pv[ib], pv[ia], bound)))
    cand.sort(key=lambda c: -c[0])                                    # descending pressure
    cp = np.array([c[0] for c in cand])
    ct = np.array([c[1] for c in cand])
    cd = np.array([c[2] for c in cand])
    theta_e = th.equivalent_potential_temperature(cp, ct, cd)
    if np.isnan(theta_e).any():
        return None
    i = int(np.argmin(theta_e))                                       # the first minimum: the larger pressure
    return cp[i], ct[i], cd[i], valid[pv >= cp[i]]


def downdraft_cape(pressure, temperature, dewpoint, opts):
    """Returns dict(dcape, downdraft_start_pressure, downdraft_start_temperature [N],
    downdraft_parcel_temperature [L, N]).  ``opts`` is an ``oracle.parcel.Options``."""
    t = np.asarray(temperature, dtype=np.float64)
    td = np.asarray(dewpoint, dtype=np.float64)
    L, N = t.shape
    p = np.broadcast_to(op._as2d(pressure), (L, N))
    ps, ts, ds = np.full(N, np.nan), np.full(N, np.nan), np.full(N, np.nan)
    descent = np.zeros((L, N), dtype=bool)
    for c in range(N):
        s = _start(p[:, c], t[:, c], td[:, c])
        if s is not None:
            ps[c], ts[c], ds[c] = s[:3]
            descent[s[3], c] = True
    ok = ~np.isnan(ps)
    # step 4: Normand wet bulb at the start point
    tw = np.full(N, np.nan)
    tw[ok] = op.wet_bulb_temperature(ps[ok], ts[ok], ds[ok], opts)
    ok &= ~np.isnan(tw)
    # step 5: the moist adiabat through (p_s, T_w); row 0 (at p_s itself) is NaN when the table has no adiabat there
    at = np.vstack([ps[None, :], np.where(descent, p, np.nan)])
    trace = np.full((L + 1, N), np.nan)
    if ok.any():
        trace[:, ok] = op._quiet(opts.moist_lapse, at[:, ok], tw[ok], ps[ok])
    ok &= ~np.isnan(trace[0])
    parcel_t = np.where(descent & ok[None, :], trace[1:], np.nan)
    # steps 6-7
    dcape = np.full(N, np.nan)
    with np.errstate(all="ignore"):
        tv_env = th.virtual_temperature(t, th.mixing_ratio_from_t_td(t, td, p, opts.metpy_compat))
        tv_par = th.virtual_temperature(parcel_t, th.saturation_mixing_ratio(p, parcel_t))
        diff = tv_env - tv_par
        for c in np.flatnonzero(ok):
            sel = descent[:, c]
            dcape[c] = -(th.RD * np.trapezoid(diff[sel, c], np.log(p[sel, c])))
    return {"dcape": dcape,
            "downdraft_start_pressure": np.where(ok, ps, np.nan),
            "downdraft_start_temperature": np.where(ok, tw, np.nan),
            "downdraft_parcel_temperature": parcel_t}


def conv_properties(dat, opts, min_set=False, downdraft=False):
    """``oracle.parcel.conv_properties`` with the ``downdraft`` keyword of the library's conv_properties: with True,
    ``dcape`` of the dewpoint derived from the specific humidity, masked like the other outputs."""
    out = op.conv_properties(dat, opts, min_set=min_set)
    if downdraft:
        p, t, q = dat["pressure"], dat["temperature"], dat["specific_humidity"]
        td = th.dewpoint_from_specific_humidity(p, t, q, opts.metpy_compat)
        dcape = downdraft_cape(p, t, td, opts)["dcape"]
        if not min_set:
            valid = ~(np.isnan(td).any(0) | np.isnan(p).any(0) | np.isnan(t).any(0) | np.isnan(q).any(0))
            dcape = np.where(valid, dcape, np.nan)
        out["dcape"] = dcape
    return out


def assert_matches(got, ora, p_max, p_start, rtol=1e-9, tie_fraction=1e-3, step_k=0.05):
    """``got`` against the oracle ``ora`` (dicts of the downdraft outputs): NaN patterns identical, every value within
    ``rtol`` relative (1 J/kg, 1 K or 1 hPa floor).  At most ``tie_fraction`` of the columns may differ by more, and
    only as a table-cell tie at one lookup does: the start temperature and the parcel by at most one adiabat step
    (``step_k``), dcape by at most Rd * 1.5 * step_k * ln(p_max / p_start) (the 1.5 covers the virtual-temperature
    factor of the saturated parcel)."""
    n = ora["dcape"].shape[0]
    bad = np.zeros(n, dtype=bool)
    for k, b in ora.items():
        if k not in got:
            continue
        a = np.asarray(got[k], dtype=np.float64)
        assert np.array_equal(np.isnan(a), np.isnan(b)), f"{k}: NaN pattern differs"
        with np.errstate(invalid="ignore"):
            err = np.where(np.isnan(b), 0.0, np.abs(a - b) / np.maximum(np.abs(b), 1.0))
        bad |= (err > rtol).reshape(-1, n).any(axis=0)
    assert bad.sum() <= tie_fraction * n, f"{bad.sum()} of {n} columns differ"
    if bad.any():
        assert np.array_equal(got["downdraft_start_pressure"][bad], ora["downdraft_start_pressure"][bad])
        assert np.all(np.abs(got["downdraft_start_temperature"][bad] - ora["downdraft_start_temperature"][bad]) <= step_k)
        bound = th.RD * 1.5 * step_k * np.log(p_max[bad] / p_start[bad])
        assert np.all(np.abs(got["dcape"][bad] - ora["dcape"][bad]) <= bound)
    return int(bad.sum())
