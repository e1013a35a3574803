"""NumPy float64 restatement of the effective inflow layer (DESIGN.md section 3.13), the reference the effective-layer
kernels are tested against.  Every lift is ``oracle.parcel``'s: the lift from level k is the most-unstable recipe
(``from_most_unstable_parcel``: keep p <= p_k, ``dropna_all``, ``shift_out_nans``, then ``cape_cin``) with its level
forced to k, vectorised over the columns; the gate is ``most_unstable_cape_cin``.  It lives beside the tests and
leaves the ``oracle`` package, which the other tests pin, unchanged.

Arrays are level-major ``[L, N]`` (level 0 = surface, pressure decreasing with the level index); pressure may be a
shared ``[L]`` axis.  ``kwargs`` are cape_cin's options (virtual_temperature_correction, lcl_interp,
pos_cape_neg_cin, post_zero_cin); ``opts`` is an ``oracle.parcel.Options`` (its metpy_compat and moist adiabat)."""

import numpy as np

from oracle import parcel as op


def valid_levels(pressure, temperature, dewpoint):
    t = np.asarray(temperature, dtype=np.float64)
    p = np.broadcast_to(op._as2d(pressure), t.shape)
    return ~(np.isnan(p) | np.isnan(t) | np.isnan(np.asarray(dewpoint, dtype=np.float64)))


def level_cape_cin(pressure, temperature, dewpoint, opts, **kwargs):
    """CAPE and CIN [L, N] of the parcel of every valid level (contract item 2); NaN on invalid levels."""
    t = np.asarray(temperature, dtype=np.float64)
    td = np.asarray(dewpoint, dtype=np.float64)
    L, N = t.shape
    p = np.array(np.broadcast_to(op._as2d(pressure), (L, N)))
    valid = valid_levels(p, t, td)
    cape, cin = np.full((L, N), np.nan), np.full((L, N), np.nan)
    for k in range(L):
        cols = np.flatnonzero(valid[k])
        if cols.size == 0:
            continue
        pc, tc, dc = p[:, cols], t[:, cols], td[:, cols]
        with np.errstate(invalid="ignore"):
            keep = pc <= pc[k][None, :]
        dat = {"pressure": np.where(keep, pc, np.nan), "temperature": np.where(keep, tc, np.nan),
               "dewpoint": np.where(keep, dc, np.nan)}
        dat, _ = op.dropna_all(dat)
        dat = op.shift_out_nans(dat, "pressure")
        res, _ = op.cape_cin(dat["pressure"], dat["temperature"], dat["dewpoint"], parcel_temperature=tc[k],
                             parcel_pressure=pc[k], parcel_dewpoint=dc[k], opts=opts, **kwargs)
        cape[k, cols] = res["cape"]
        cin[k, cols] = res["cin"]
    return cape, cin


def passes(cape, cin, min_cape=100.0, min_cin=-250.0):
    with np.errstate(invalid="ignore"):
        return (cape >= min_cape) & (cin > min_cin)


def gate(pressure, temperature, dewpoint, opts, min_cape=100.0, min_cin=-250.0, depth=300.0, **kwargs):
    """Contract item 4: the most-unstable parcel passes [N]."""
    t = np.asarray(temperature, dtype=np.float64)
    p = np.array(np.broadcast_to(op._as2d(pressure), t.shape))
    res, _, _ = op.most_unstable_cape_cin(p, t, dewpoint, opts, depth=depth, **kwargs)
    return passes(res["cape"], res["cin"], min_cape, min_cin)


def search(level_cape, level_cin, gate_ok, valid, min_cape=100.0, min_cin=-250.0):
    """Contract items 5-6 on per-level values [L, N]: (base level, top level) [N], -1 where there is none."""
    L, N = level_cape.shape
    ok = passes(level_cape, level_cin, min_cape, min_cin)
    base, top = np.full(N, -1), np.full(N, -1)
    for c in np.flatnonzero(gate_ok):
        ks = np.flatnonzero(valid[:, c])
        hit = ks[ok[ks, c]]
        if hit.size == 0:
            continue
        base[c] = hit[0]
        above = ks[ks > hit[0]]
        fail = above[~ok[above, c]]
        if fail.size:
            top[c] = above[above < fail[0]].max(initial=hit[0])
    return base, top


def level_pressure(pressure, shape, k):
    """The input pressure of level k[c] of each column, NaN where k is -1."""
    p = np.broadcast_to(op._as2d(pressure), shape)
    n = np.arange(shape[1])
    return np.where(k >= 0, p[np.maximum(k, 0), n], np.nan)


def effective_inflow_layer(pressure, temperature, dewpoint, opts, min_cape=100.0, min_cin=-250.0, depth=300.0,
                           **kwargs):
    """dict(effective_inflow_base, effective_inflow_top [N], level_parcel_cape, level_parcel_cin [L, N],
    gate [N])."""
    t = np.asarray(temperature, dtype=np.float64)
    cape, cin = level_cape_cin(pressure, t, dewpoint, opts, **kwargs)
    g = gate(pressure, t, dewpoint, opts, min_cape, min_cin, depth, **kwargs)
    base, top = search(cape, cin, g, valid_levels(pressure, t, dewpoint), min_cape, min_cin)
    return {"effective_inflow_base": level_pressure(pressure, t.shape, base),
            "effective_inflow_top": level_pressure(pressure, t.shape, top),
            "level_parcel_cape": cape, "level_parcel_cin": cin, "gate": g}
