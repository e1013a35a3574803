// xp_kinematics.cuh -- Bunkers storm motion, storm-relative helicity and bulk wind difference of one column, and the
// effective-layer supercell / tornado composites of one point (DESIGN.md section 3.14).  Host-compilable for
// tests/hostsim (see xp_math.cuh).  float64 arithmetic in the order written here (no FMA contraction).
//
// Wind profile of a column: the surface point (z = 0, su, sv), then, in level order, every level whose height z (m
// above the surface), u and v are all non-NaN and whose z > 0.  A NaN surface wind, or kept heights that do not
// increase strictly, make every output of the column NaN.  V(z) is the profile interpolated linearly in height; a
// profile point exactly at z is used as it is.
//
// Layer [a, b] (a bound below 0 is taken as 0): its points are a, the profile points strictly inside (a, b), and b.
// It is NaN if a or b is NaN, if b < a, or if b lies above the highest profile point read.
//   mean wind = trapezoid(V, z) / (b - a);   BWD = V(b) - V(a);
//   SRH(c)    = sum_i (u_{i+1} - c_u)(v_i - c_v) - (u_i - c_u)(v_{i+1} - c_v), which telescopes to
//               S + c_v (u_a - u_b) + c_u (v_b - v_a) with S = sum_i u_{i+1} v_i - u_i v_{i+1}: one upward pass
//               accumulates S and the end winds of every layer, and the storm motion c is applied after it.
// Bunkers motion (Bunkers et al. 2000): M = mean wind over [0, 6000], S = mean over [5500, 6000] - mean over [0, 500],
// right / left = M +- 7.5 (S_v, -S_u) / |S|; NaN when |S| == 0 or a layer is NaN.  SRH is NaN where the motion is.
//
// The column is read in level order up to the first profile point at or above the highest bound the call needs (6000 m
// when it asks for Bunkers motion or any SRH) and no further; the strictly-increasing check covers those points.
#pragma once
#include "xp_math.cuh"

namespace xp {

constexpr int kMaxSrhDepths = 4;
constexpr double kBunkersDeviation = 7.5;          // m/s

// What one call computes (the same for every column).
struct KinematicsRequest {
    bool motion;                      // Bunkers motion (needed by every SRH)
    int n_depths;                     // SRH over [0, depth[j]], j < n_depths
    double depth[kMaxSrhDepths];
    bool srh_layer, bwd_layer;        // the per-column layers
    double mover;                     // +1 right, -1 left
};

struct KinematicsResult {
    double right_u, right_v, left_u, left_v, mean_u, mean_v;
    double srh[kMaxSrhDepths];
    double srh_layer;
    double bwd_u, bwd_v, bwd_magnitude;
};

// One layer's accumulators over the upward pass.  Fields a layer kind never reads are dead and compile away.
struct KinLayer {
    double a, b;                      // bounds, a >= 0; NaN: the layer is not computed
    double iu, iv;                    // trapezoid(V, z)
    double s;                         // sum u_{i+1} v_i - u_i v_{i+1}
    double ua, va, ub, vb;            // V(a), V(b)
    bool done;

    XP_HD void init(double lo, double hi) {
        lo = lo < 0.0 ? 0.0 : lo;                                   // NaN stays NaN
        hi = hi < 0.0 ? 0.0 : hi;
        a = lo; b = hi;
        iu = iv = s = 0.0;
        ua = va = ub = vb = qnan();
        done = isnan(lo) || isnan(hi) || hi < lo;                   // NaN layer: never accumulates
        if (done) a = b = qnan();
    }
    XP_HD bool ok() const { return done && !isnan(b); }

    // the profile segment (z0, u0, v0) -> (z1, u1, v1), z0 < z1; z0 = z1 for the surface point alone
    XP_HD void segment(double z0, double u0, double v0, double z1, double u1, double v1) {
        if (done) return;
        if (a < z1 && b > z0) {
            double us = u0, vs = v0, zs = z0;
            if (a > z0) {
                zs = a;
                us = u0 + (a - z0) * (u1 - u0) / (z1 - z0);
                vs = v0 + (a - z0) * (v1 - v0) / (z1 - z0);
            }
            if (a >= z0) { ua = us; va = vs; }
            double ue = u1, ve = v1, ze = z1;
            if (b < z1) {
                ze = b;
                ue = u0 + (b - z0) * (u1 - u0) / (z1 - z0);
                ve = v0 + (b - z0) * (v1 - v0) / (z1 - z0);
            }
            iu += (ze - zs) * (us + ue) / 2.0;
            iv += (ze - zs) * (vs + ve) / 2.0;
            s += ue * vs - us * ve;
            if (b <= z1) { ub = ue; vb = ve; done = true; }
        } else if (b <= z1) {                       // zero-depth layer at exactly the profile point z1
            ua = ub = u1; va = vb = v1;
            done = true;
        }
    }
    XP_HD double srh(double cu, double cv) const {
        if (!ok()) return qnan();
        return s + cv * (ua - ub) + cu * (vb - va);
    }
};

// The whole column.  `load(k, z, u, v)` reads level k.  sb / st: the SRH layer, bb / bt: the BWD layer (ignored
// unless requested).
template <class Load>
XP_HD void storm_kinematics(int L, Load load, double su, double sv, const KinematicsRequest &rq, double sb, double st,
                            double bb, double bt, KinematicsResult &r) {
    const double nan = qnan();
    r.right_u = r.right_v = r.left_u = r.left_v = r.mean_u = r.mean_v = nan;
    for (int j = 0; j < kMaxSrhDepths; ++j) r.srh[j] = nan;
    r.srh_layer = r.bwd_u = r.bwd_v = r.bwd_magnitude = nan;
    if (isnan(su) || isnan(sv)) return;
    const bool motion = rq.motion || rq.n_depths > 0 || rq.srh_layer;
    KinLayer low, high, deep, dep[kMaxSrhDepths], sl, bl;
    low.init(motion ? 0.0 : nan, 500.0);
    high.init(motion ? 5500.0 : nan, 6000.0);
    deep.init(motion ? 0.0 : nan, 6000.0);
#pragma unroll
    for (int j = 0; j < kMaxSrhDepths; ++j) dep[j].init(j < rq.n_depths ? 0.0 : nan, rq.depth[j]);
    sl.init(rq.srh_layer ? sb : nan, st);
    bl.init(rq.bwd_layer ? bb : nan, bt);
    auto all_done = [&]() {
        bool d = low.done && high.done && deep.done && sl.done && bl.done;
#pragma unroll
        for (int j = 0; j < kMaxSrhDepths; ++j) d = d && dep[j].done;
        return d;
    };
    auto step = [&](double z0, double u0, double v0, double z1, double u1, double v1) {
        low.segment(z0, u0, v0, z1, u1, v1);
        high.segment(z0, u0, v0, z1, u1, v1);
        deep.segment(z0, u0, v0, z1, u1, v1);
#pragma unroll
        for (int j = 0; j < kMaxSrhDepths; ++j) dep[j].segment(z0, u0, v0, z1, u1, v1);
        sl.segment(z0, u0, v0, z1, u1, v1);
        bl.segment(z0, u0, v0, z1, u1, v1);
    };
    double z0 = 0.0, u0 = su, v0 = sv;
    step(z0, u0, v0, z0, u0, v0);                   // layers that end at the surface
    for (int k = 0; k < L && !all_done(); ++k) {
        double z, u, v;
        load(k, z, u, v);
        if (isnan(z) || isnan(u) || isnan(v) || !(z > 0.0)) continue;
        if (!(z > z0)) return;                      // kept heights must increase strictly
        step(z0, u0, v0, z, u, v);
        z0 = z; u0 = u; v0 = v;
    }
    if (motion && low.ok() && high.ok() && deep.ok()) {
        const double mu = deep.iu / (deep.b - deep.a), mv = deep.iv / (deep.b - deep.a);
        const double shu = high.iu / (high.b - high.a) - low.iu / (low.b - low.a);
        const double shv = high.iv / (high.b - high.a) - low.iv / (low.b - low.a);
        const double mag = sqrt(shu * shu + shv * shv);
        if (mag != 0.0) {
            const double du = kBunkersDeviation * shv / mag, dv = -(kBunkersDeviation * shu) / mag;
            r.mean_u = mu; r.mean_v = mv;
            r.right_u = mu + du; r.right_v = mv + dv;
            r.left_u = mu - du; r.left_v = mv - dv;
        }
    }
    const double cu = rq.mover > 0.0 ? r.right_u : r.left_u;
    const double cv = rq.mover > 0.0 ? r.right_v : r.left_v;
    for (int j = 0; j < kMaxSrhDepths; ++j)
        if (j < rq.n_depths) r.srh[j] = dep[j].srh(cu, cv);
    if (rq.srh_layer) r.srh_layer = sl.srh(cu, cv);
    if (rq.bwd_layer && bl.ok()) {
        r.bwd_u = bl.ub - bl.ua;
        r.bwd_v = bl.vb - bl.va;
        r.bwd_magnitude = sqrt(r.bwd_u * r.bwd_u + r.bwd_v * r.bwd_v);
    }
}

// np.maximum(0, x): NaN propagates
XP_HD double kin_max0(double x) { return isnan(x) ? x : (0.0 >= x ? 0.0 : x); }

// Supercell composite parameter (SHARPpy params.scp): J/kg, m2/s2, m/s.
XP_HD double supercell_composite(double mucape, double esrh, double ebwd) {
    const double tb = isnan(ebwd) ? ebwd : (ebwd < 10.0 ? 0.0 : (ebwd > 20.0 ? 1.0 : ebwd / 20.0));
    return (mucape / 1000.0) * (esrh / 50.0) * tb;
}

// Effective-layer significant tornado parameter with CIN (SHARPpy params.stp_cin): J/kg, m2/s2, m/s, m AGL, J/kg.
XP_HD double significant_tornado(double mlcape, double esrh, double ebwd, double lcl_h, double mlcin) {
    const double tb = isnan(ebwd) ? ebwd : (ebwd < 12.5 ? 0.0 : (ebwd > 30.0 ? 1.5 : ebwd / 20.0));
    const double tl = isnan(lcl_h) ? lcl_h : (lcl_h < 1000.0 ? 1.0 : (lcl_h > 2000.0 ? 0.0 : (2000.0 - lcl_h) / 1000.0));
    const double tc = isnan(mlcin) ? mlcin : (mlcin > -50.0 ? 1.0 : (mlcin < -200.0 ? 0.0 : (mlcin + 200.0) / 150.0));
    return kin_max0((mlcape / 1500.0) * (esrh / 150.0) * tb * tl * tc);
}

}  // namespace xp
