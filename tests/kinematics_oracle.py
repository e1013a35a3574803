"""NumPy float64 restatement of the storm kinematics, the supercell / tornado composites and the effective-layer
composition (DESIGN.md section 3.14) in their direct form, the reference the kinematics kernels are tested against.

Each layer's point list is built explicitly (its bottom, the profile points strictly inside, its top); the mean wind
is ``np.trapezoid`` over it and SRH is MetPy's ``storm_relative_helicity`` sum over consecutive points.  The column
code accumulates a ground-relative sum and applies the storm motion after one pass instead, so the two agree to
rounding, not bit for bit.  The effective composition is built on ``effective_oracle`` and ``oracle.parcel``.

Arrays are level-major ``[L, N]`` (level 0 = surface); heights are m above the surface."""

import numpy as np

import effective_oracle as eo
from oracle import parcel as op

def profile(z, u, v, su, sv, top):
    """The wind profile of one column read up to the first point at or above ``top`` (NaN: read every level):
    arrays (z, u, v) starting with the surface point, or None when the column's outputs are all NaN."""
    if np.isnan(su) or np.isnan(sv):
        return None
    zs, us, vs = [0.0], [float(su)], [float(sv)]
    for k in range(len(z)):
        if not np.isnan(top) and zs[-1] >= top:
            break
        if np.isnan(z[k]) or np.isnan(u[k]) or np.isnan(v[k]) or not z[k] > 0.0:
            continue
        if not z[k] > zs[-1]:
            return None
        zs.append(float(z[k]))
        us.append(float(u[k]))
        vs.append(float(v[k]))
    return np.array(zs), np.array(us), np.array(vs)


def at(prof, x):
    """V(x): a profile point exactly at x as it is, else linear in height between its neighbours."""
    z, u, v = prof
    j = int(np.searchsorted(z, x, side="left"))
    if z[j] == x:
        return u[j], v[j]
    d = z[j] - z[j - 1]
    return (u[j - 1] + (x - z[j - 1]) * (u[j] - u[j - 1]) / d, v[j - 1] + (x - z[j - 1]) * (v[j] - v[j - 1]) / d)


def layer(prof, a, b):
    """The layer's points (z, u, v) over [a, b], or None when the layer is NaN."""
    if prof is None or np.isnan(a) or np.isnan(b):
        return None
    a, b = max(a, 0.0), max(b, 0.0)
    z, u, v = prof
    if b < a or b > z[-1]:
        return None
    inside = (z > a) & (z < b)
    ua, va = at(prof, a)
    ub, vb = at(prof, b)
    return (np.concatenate([[a], z[inside], [b]]), np.concatenate([[ua], u[inside], [ub]]),
            np.concatenate([[va], v[inside], [vb]]))


def mean_wind(pts):
    z, u, v = pts
    return np.trapezoid(u, z) / (z[-1] - z[0]), np.trapezoid(v, z) / (z[-1] - z[0])


def srh_terms(pts, cu, cv):
    """MetPy's storm-relative helicity terms over consecutive layer points."""
    _, u, v = pts
    su, sv = u - cu, v - cv
    return su[1:] * sv[:-1] - su[:-1] * sv[1:]


def bunkers(prof):
    """(right_u, right_v, left_u, left_v, mean_u, mean_v), NaN where undefined."""
    nan6 = (np.nan,) * 6
    lays = [layer(prof, 0.0, 6000.0), layer(prof, 5500.0, 6000.0), layer(prof, 0.0, 500.0)]
    if any(x is None for x in lays):
        return nan6
    mu, mv = mean_wind(lays[0])
    hu, hv = mean_wind(lays[1])
    lu, lv = mean_wind(lays[2])
    shu, shv = hu - lu, hv - lv
    mag = np.sqrt(shu * shu + shv * shv)
    if mag == 0.0:
        return nan6
    du, dv = 7.5 * shv / mag, -7.5 * shu / mag
    return mu + du, mv + dv, mu - du, mv - dv, mu, mv


def storm_kinematics(z, u, v, su, sv, mover=1, depths=(), srh_layer=None, bwd_layer=None, motion=True):
    """The kinematics entry on [L, N] columns, every output computed.  Returns (dict of [N] outputs, dict of [N]
    absolute-term scales for the tolerance ``1 + sum |terms|``).  ``motion``: the call asks for the motion (it sets the
    read extent with the depths and layers, as the C entry does)."""
    z, u, v = [np.asarray(x, np.float64) for x in (z, u, v)]
    L, N = z.shape
    su = np.broadcast_to(np.asarray(su, np.float64), (N,))
    sv = np.broadcast_to(np.asarray(sv, np.float64), (N,))
    names = ["bunkers_right_u", "bunkers_right_v", "bunkers_left_u", "bunkers_left_v", "mean_wind_u", "mean_wind_v"]
    out = {n: np.full(N, np.nan) for n in names}
    scale = {n: np.ones(N) for n in names}
    dn = [f"srh_0_{float(d):g}m" for d in depths]
    extra = dn + (["srh_layer"] if srh_layer is not None else []) + \
        (["bulk_wind_difference_u", "bulk_wind_difference_v", "bulk_wind_difference"] if bwd_layer is not None else [])
    for n in extra:
        out[n] = np.full(N, np.nan)
        scale[n] = np.ones(N)
    need_motion = motion or len(depths) > 0 or srh_layer is not None
    for c in range(N):
        tops = ([6000.0] if need_motion else []) + [float(d) for d in depths]
        lay_s = lay_b = None
        if srh_layer is not None:
            lay_s = (float(srh_layer[0][c]), float(srh_layer[1][c]))
        if bwd_layer is not None:
            lay_b = (float(bwd_layer[0][c]), float(bwd_layer[1][c]))
        for lb in (lay_s, lay_b):
            if lb is not None and not (np.isnan(lb[0]) or np.isnan(lb[1])) and max(lb[1], 0.0) >= max(lb[0], 0.0):
                tops.append(max(lb[1], 0.0))
        top = max(tops) if tops else -1.0
        prof = profile(z[:, c], u[:, c], v[:, c], su[c], sv[c], top) if top >= 0.0 else None
        mot = bunkers(prof) if need_motion and prof is not None else (np.nan,) * 6
        for n, x in zip(names, mot):
            out[n][c] = x
        if need_motion and prof is not None:
            for lo, hi in ((0.0, 6000.0), (5500.0, 6000.0), (0.0, 500.0)):
                pts = layer(prof, lo, hi)
                if pts is not None:
                    s = np.abs(pts[1]).sum() + np.abs(pts[2]).sum() + 7.5
                    for n in names:
                        scale[n][c] = max(scale[n][c], 1.0 + s)
        cu, cv = (mot[0], mot[1]) if mover > 0 else (mot[2], mot[3])

        def srh(a, b):
            pts = layer(prof, a, b)
            if pts is None or np.isnan(cu):
                return np.nan, 1.0
            # scale: the products of either form (storm-relative terms, or ground-relative terms plus the motion's)
            m = np.abs(pts[1]) + np.abs(pts[2]) + abs(cu) + abs(cv)
            return float(srh_terms(pts, cu, cv).sum()), 1.0 + float((m[1:] * m[:-1]).sum())
        for n, d in zip(dn, depths):
            out[n][c], scale[n][c] = srh(0.0, float(d))
        if lay_s is not None:
            out["srh_layer"][c], scale["srh_layer"][c] = srh(*lay_s)
        if lay_b is not None:
            pts = layer(prof, *lay_b)
            if pts is not None:
                du, dv = pts[1][-1] - pts[1][0], pts[2][-1] - pts[2][0]
                out["bulk_wind_difference_u"][c], out["bulk_wind_difference_v"][c] = du, dv
                out["bulk_wind_difference"][c] = np.sqrt(du * du + dv * dv)
                s = 1.0 + abs(pts[1][0]) + abs(pts[1][-1]) + abs(pts[2][0]) + abs(pts[2][-1])
                for n in ("bulk_wind_difference_u", "bulk_wind_difference_v", "bulk_wind_difference"):
                    scale[n][c] = s
    return out, scale


def supercell_composite(mucape, esrh, ebwd):
    """SHARPpy ``params.scp``, NaN in giving NaN out."""
    mucape, esrh, ebwd = np.broadcast_arrays(*[np.asarray(x, np.float64) for x in (mucape, esrh, ebwd)])
    with np.errstate(invalid="ignore"):
        tb = np.where(ebwd < 10.0, 0.0, np.where(ebwd > 20.0, 1.0, ebwd / 20.0))
    tb = np.where(np.isnan(ebwd), np.nan, tb)
    return (mucape / 1000.0) * (esrh / 50.0) * tb


def significant_tornado(mlcape, esrh, ebwd, lcl_height, mlcin):
    """SHARPpy ``params.stp_cin``, NaN in giving NaN out (``np.maximum``)."""
    mlcape, esrh, ebwd, lcl_height, mlcin = np.broadcast_arrays(
        *[np.asarray(x, np.float64) for x in (mlcape, esrh, ebwd, lcl_height, mlcin)])
    with np.errstate(invalid="ignore"):
        tb = np.where(ebwd < 12.5, 0.0, np.where(ebwd > 30.0, 1.5, ebwd / 20.0))
        tl = np.where(lcl_height < 1000.0, 1.0, np.where(lcl_height > 2000.0, 0.0, (2000.0 - lcl_height) / 1000.0))
        tc = np.where(mlcin > -50.0, 1.0, np.where(mlcin < -200.0, 0.0, (mlcin + 200.0) / 150.0))
    tb = np.where(np.isnan(ebwd), np.nan, tb)
    tl = np.where(np.isnan(lcl_height), np.nan, tl)
    tc = np.where(np.isnan(mlcin), np.nan, tc)
    return np.maximum(0.0, (mlcape / 1500.0) * (esrh / 150.0) * tb * tl * tc)


def lifts(pressure, temperature, dewpoint, opts, mixed_layer_depth=100.0, most_unstable_depth=300.0, **kwargs):
    """The pieces the composition takes from the ML and MU lifts [N]."""
    t = np.asarray(temperature, np.float64)
    p = np.array(np.broadcast_to(op._as2d(pressure), t.shape))
    ml, ml_prof, _ = op.mixed_layer_cape_cin(p, t, dewpoint, opts, depth=mixed_layer_depth, **kwargs)
    mu, mu_prof, _ = op.most_unstable_cape_cin(p, t, dewpoint, opts, depth=most_unstable_depth, **kwargs)
    return {"mu_cape": mu["cape"], "mu_el_pressure": mu_prof["el_pressure"], "ml_cape": ml["cape"],
            "ml_cin": ml["cin"], "ml_lcl_pressure": ml_prof["lcl_pressure"]}


def effective_layer_parameters(pressure, temperature, dewpoint, height, wind_u, wind_v, surface_wind_u,
                               surface_wind_v, opts, mover=1, min_cape=100.0, min_cin=-250.0,
                               most_unstable_depth=300.0, mixed_layer_depth=100.0, pieces=None, **kwargs):
    """The effective-layer composition.  ``pieces``: the base / top pressures and the lift values (``lifts``'s keys
    plus effective_inflow_base / _top) to compose from instead of computing them here.  Returns (outputs, scales,
    the pieces with the heights z_base, z_top, z_el, z_lcl; computed here, the pieces include the effective layer's
    level_parcel_cape / _cin)."""
    t = np.asarray(temperature, np.float64)
    L, N = t.shape
    p = np.array(np.broadcast_to(op._as2d(pressure), (L, N)))
    if pieces is None:
        eff = eo.effective_inflow_layer(p, t, dewpoint, opts, min_cape, min_cin, most_unstable_depth, **kwargs)
        pieces = dict(lifts(p, t, dewpoint, opts, mixed_layer_depth, most_unstable_depth, **kwargs),
                      **{k: eff[k] for k in ("effective_inflow_base", "effective_inflow_top", "level_parcel_cape",
                                             "level_parcel_cin")})
    h = np.asarray(height, np.float64)

    def z_at(pr):
        return op.log_interp({"h": h}, p, np.asarray(pr, np.float64))["h"]

    zb, zt = z_at(pieces["effective_inflow_base"]), z_at(pieces["effective_inflow_top"])
    zel, zlcl = z_at(pieces["mu_el_pressure"]), z_at(pieces["ml_lcl_pressure"])
    zb0 = np.maximum(zb, 0.0)
    mid = zb0 + (zel - zb0) / 2.0
    kin, sc = storm_kinematics(h, wind_u, wind_v, surface_wind_u, surface_wind_v, mover, srh_layer=(zb, zt),
                               bwd_layer=(zb0, mid), motion=False)
    esrh, ebwd = kin["srh_layer"], kin["bulk_wind_difference"]
    no_layer = np.isnan(np.asarray(pieces["effective_inflow_base"], np.float64))
    esrh = np.where(no_layer, np.nan, esrh)
    ebwd = np.where(no_layer, np.nan, ebwd)
    s_in = np.where(no_layer, 0.0, esrh) * mover
    b_in = np.where(no_layer, 0.0, ebwd)
    out = {"effective_inflow_base": np.asarray(pieces["effective_inflow_base"], np.float64),
           "effective_inflow_top": np.asarray(pieces["effective_inflow_top"], np.float64),
           "effective_srh": esrh, "effective_bulk_wind_difference": ebwd,
           "supercell_composite_parameter": supercell_composite(pieces["mu_cape"], s_in, b_in),
           "significant_tornado_parameter": significant_tornado(pieces["ml_cape"], s_in, b_in, zlcl, pieces["ml_cin"])}
    scales = {"effective_srh": sc["srh_layer"], "effective_bulk_wind_difference": sc["bulk_wind_difference"]}
    return out, scales, dict(pieces, z_base=zb, z_top=zt, z_el=zel, z_lcl=zlcl)
