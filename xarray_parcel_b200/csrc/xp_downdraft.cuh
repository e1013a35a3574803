// xp_downdraft.cuh -- downdraft CAPE (DCAPE) of one column, MetPy's downdraft_cape recipe on this project's
// thermodynamics and lookup-table moist adiabat (DESIGN.md section 3.12).  Host-compilable for tests/hostsim
// (see xp_math.cuh).
//
// Per column, levels numbered from the surface, pressure decreasing with the level index:
//   1. a level is valid when p, T and Td are all non-NaN; invalid levels are skipped everywhere;
//   2. candidates: the valid levels in 700..500 hPa (np.isclose to a bound counts as inside), plus a point at
//      exactly 700 / 500 hPa interpolated in ln p between the bracketing valid levels when no valid level is close
//      to that bound; a column that cannot bracket both bounds gives NaN everywhere;
//   3. start = the candidate of minimum theta-e (Bolton), the first one (larger pressure) on a tie; a NaN theta-e
//      gives NaN everywhere;
//   4. T_w = Normand wet bulb at the start (lcl_solve, then the adiabat of the LCL's table cell at p_s);
//   5. the parcel descends on adiabat adiabat_lookup(p_s, T_w) to every valid level with p >= p_s; a table index
//      of 0 at either lookup gives NaN everywhere;
//   6. d = Tv_env - Tv_parcel with the virtual temperatures of parcel_profile_with_lcl (PF:684-710, 760, 782-804);
//   7. dcape = -(Rd * trapezoid(d, ln p)) over the descent levels, surface first; NaN anywhere gives NaN.
#pragma once
#include "xp_column.cuh"

namespace xp {

constexpr double kDowndraftBottom = 700.0;     // hPa, layer searched for the downdraft source
constexpr double kDowndraftTop = 500.0;

struct DowndraftResult {
    double dcape, p_start, t_start;
    int k_end;          // last level index of the descent (valid levels 0..k_end with p >= p_start), -1 on failure
    int adiabat;        // 1-based descent adiabat, 0 on failure
};

// np.isclose(p, bound) with the default tolerances
XP_HD bool dd_close(double p, double bound) { return fabs(p - bound) <= 1e-8 + 1e-5 * bound; }

// v_b + (ln x - ln p_b) (v_a - v_b) / (ln p_a - ln p_b): b = the bracketing valid level of larger pressure
XP_HD double dd_interp(double vb, double va, double lpb, double lpa, double lx) {
    return vb + (lx - lpb) * (va - vb) / (lpa - lpb);
}

// Steps 1-5: the start point and the descent adiabat.  `load(k, p, t, td)` reads level k.  Reads levels from the
// surface up to the first valid level beyond the 500 hPa bound and no further.
template <class Load>
XP_HD void downdraft_start(int L, Load load, const Tables &tb, DowndraftResult &r) {
    r.dcape = r.p_start = r.t_start = qnan();
    r.k_end = -1;
    r.adiabat = 0;
    bool have_prev = false, seen700 = false, seen500 = false, done = false, fail = false;
    int k_prev = -1;
    double pp = qnan(), tp = qnan(), dp = qnan();
    double best = qnan(), ps = qnan(), ts = qnan(), ds = qnan();
    int k_start = -1;
    bool any = false;
    auto candidate = [&](double p, double t, double td, int k_desc) {
        const double th = theta_e(p, t, td);
        if (isnan(th)) { fail = true; return; }
        if (!any || th < best) { best = th; ps = p; ts = t; ds = td; k_start = k_desc; }
        any = true;
    };
    for (int k = 0; k < L && !done && !fail; ++k) {
        double p, t, td;
        load(k, p, t, td);
        if (isnan(p) || isnan(t) || isnan(td)) continue;
        const bool c700 = dd_close(p, kDowndraftBottom), c500 = dd_close(p, kDowndraftTop);
        if (c700) seen700 = true;
        if (!seen700 && p < kDowndraftBottom) {
            // first valid level below 700 hPa with none close to it: the interpolated point at 700 (or no bracket)
            if (!have_prev) { fail = true; break; }
            const double lb = xp_log(pp), la = xp_log(p), lx = xp_log(kDowndraftBottom);
            candidate(kDowndraftBottom, dd_interp(tp, t, lb, la, lx), dd_interp(dp, td, lb, la, lx), k_prev);
            seen700 = true;
            if (fail) break;
        }
        if ((p <= kDowndraftBottom || c700) && (p >= kDowndraftTop || c500)) {
            candidate(p, t, td, k);
            if (c500) seen500 = true;
        } else if (p < kDowndraftTop) {
            // first valid level beyond the 500 hPa bound: the interpolated point at 500 when no level is close to it
            if (!seen500) {
                const double lb = xp_log(pp), la = xp_log(p), lx = xp_log(kDowndraftTop);
                candidate(kDowndraftTop, dd_interp(tp, t, lb, la, lx), dd_interp(dp, td, lb, la, lx), k_prev);
                seen500 = true;
            }
            done = true;
        }
        have_prev = true; k_prev = k; pp = p; tp = t; dp = td;
    }
    if (fail || !seen500 || !any) return;
    double lcl_p, lcl_t;
    lcl_solve(ps, ts, ds, lcl_p, lcl_t);
    const int a_lcl = adiabat_lookup(tb, lcl_p, lcl_t);
    if (a_lcl <= 0) return;
    const double tw = adiabat_temperature(tb.curves + (size_t)(a_lcl - 1) * kNP, ps);
    const int a = adiabat_lookup(tb, ps, tw);
    if (a <= 0) return;
    r.p_start = ps;
    r.t_start = tw;
    r.k_end = k_start;
    r.adiabat = a;
}

// Steps 6-7 on the levels 0..k_end.  `put(k, parcel_t)` receives the parcel temperature of every level 0..k_end
// (NaN on invalid levels).
template <class Load, class Put>
XP_HD void downdraft_integral(Load load, const Tables &tb, int compat, DowndraftResult &r, Put put) {
    if (r.adiabat <= 0) return;
    const float *curve = tb.curves + (size_t)(r.adiabat - 1) * kNP;
    double sum = 0.0, x0 = qnan(), d0 = qnan();
    bool first = true;
    for (int k = 0; k <= r.k_end; ++k) {
        double p, t, td;
        load(k, p, t, td);
        if (isnan(p) || isnan(t) || isnan(td)) { put(k, qnan()); continue; }
        const double tpar = adiabat_temperature(curve, p);
        put(k, tpar);
        const double tv_env = virtual_temperature(t, mixing_ratio_t_td(t, td, p, compat));
        const double tv_par = virtual_temperature(tpar, sat_mixing_ratio(p, tpar));
        const double d = tv_env - tv_par;
        const double x = xp_log(p);
        if (!first) sum += (x - x0) * (d + d0) / 2.0;          // np.trapezoid: d * (y[1:] + y[:-1]) / 2.0
        first = false;
        x0 = x; d0 = d;
    }
    r.dcape = -(kRd * sum);
}

}  // namespace xp
