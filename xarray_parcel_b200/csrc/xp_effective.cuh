// xp_effective.cuh -- the effective inflow layer (Thompson et al. 2007, SHARPpy's effective_inflow_layer) of one
// column, on this library's parcel lift (DESIGN.md section 3.13).  Host-compilable for tests/hostsim (see
// xp_math.cuh).  No new thermodynamics: every lift is lift_parcel on LiftedLevels, as in the most-unstable path.
//
// Per column, levels numbered from the surface, pressure decreasing with the level index:
//   1. a level is valid when p, T and Td are all non-NaN; only valid levels are lifted or can be a base or a top;
//   2. the lift from level k is the parcel (p_k, T_k, Td_k) on the levels with p <= p_k: the most-unstable lift
//      with its level forced to k (LiftedLevels{k0 = k, mode = 1, thresh = p_k});
//   3. a level passes when cape >= min_cape && cin > min_cin (a NaN fails);
//   4. gate: the column's most-unstable parcel (run_column kind 2, over most_unstable_depth) must pass, else base
//      and top are NaN;
//   5. base: the first valid level from the surface upward that passes (none: base and top NaN);
//   6. top: the valid level just below the first valid level above the base that fails; NaN when none fails.
#pragma once
#include "xp_parcels.cuh"

namespace xp {

struct EffNoProf {
    XP_HD void put(int, const ProfileRow &) const {}
};

XP_HD bool eff_valid(double p, double t, double td) { return !(isnan(p) || isnan(t) || isnan(td)); }
XP_HD bool eff_pass(double cape, double cin, double min_cape, double min_cin) {
    return cape >= min_cape && cin > min_cin;
}

// Item 2: the parcel of valid level k lifted over the levels with p <= p_k.
template <class Reader>
XP_HD void eff_lift(const Reader &rd, int k, const Tables &tb, const Opts &o, ParcelResult &r) {
    LiftedLevels<Reader> lv;
    lv.rd = rd; lv.k0 = k; lv.pre = 0; lv.mode = 1;
    const double p = rd.P(k);
    lv.thresh = p;
    lv.pre_p = lv.pre_t = lv.pre_td = qnan();
    EffNoProf np;
    lift_parcel(lv, p, rd.Tk(k), rd.Td(k), tb, o, r, np);
}

// Item 4 through run_column(kind = 2).  Returns the pass of the most-unstable parcel; k_mu = its level (rd.L when
// the column has none).
template <class Reader>
XP_HD bool eff_gate(const Reader &rd, const Tables &tb, const Opts &o, double min_cape, double min_cin, int &k_mu,
                    uint32_t &flags) {
    ParcelResult r;
    double p0, t0, td0;
    EffNoProf np;
    run_column(rd, 2, tb, o, qnan(), qnan(), qnan(), r, p0, t0, td0, k_mu, np);
    flags |= r.flags;
    return eff_pass(r.cape, r.cin, min_cape, min_cin);
}

// Items 5-6 as a state machine fed with the pass of each valid level, from the surface upward.
struct EffSearch {
    int state;                  // 0: looking for the base, 1: inside the layer, 2: top decided
    double base_p, top_p, last_p;
    XP_HD void init() { state = 0; base_p = top_p = last_p = qnan(); }
    XP_HD bool done() const { return state == 2; }
    XP_HD void feed(double p, bool pass) {
        if (state == 0) {
            if (pass) { state = 1; base_p = last_p = p; }
        } else if (state == 1) {
            if (pass) last_p = p;
            else { state = 2; top_p = last_p; }
        }
    }
};

// Search mode, after a gate that passed: lifts successive valid levels until the top is decided.  k_known is the
// most-unstable level, whose pass the gate has already established (the same lift, so the same bits): it is not
// lifted again.
template <class Reader>
XP_HD void eff_search(const Reader &rd, const Tables &tb, const Opts &o, double min_cape, double min_cin,
                      int k_known, uint32_t &flags, double &base_p, double &top_p) {
    EffSearch s;
    s.init();
    for (int k = 0; k < rd.L && !s.done(); ++k) {
        const double p = rd.P(k);
        if (!eff_valid(p, rd.Tk(k), rd.Td(k))) continue;
        bool pass = true;
        if (k != k_known) {
            ParcelResult r;
            eff_lift(rd, k, tb, o, r);
            flags |= r.flags;
            pass = eff_pass(r.cape, r.cin, min_cape, min_cin);
        }
        s.feed(p, pass);
    }
    base_p = s.base_p;
    top_p = s.top_p;
}

// All-levels mode: lifts every valid level, put(k, cape, cin) for every level 0..L-1 (NaN on invalid levels), and
// the same base and top as the gate and eff_search give.  The gate is read off the levels: the most-unstable lift
// IS the lift from level k_mu; a column without a most-unstable parcel lifts a NaN parcel, which lift_parcel gives
// cape = cin = 0.
template <class Reader, class Put>
XP_HD void eff_all_levels(const Reader &rd, const Tables &tb, const Opts &o, double min_cape, double min_cin,
                          uint32_t &flags, double &base_p, double &top_p, Put put) {
    double mu_p, mu_t, mu_td;
    int k_mu;
    most_unstable_parcel(rd, o.mu_depth, mu_p, mu_t, mu_td, k_mu, flags);
    bool gate = k_mu >= rd.L && eff_pass(0.0, 0.0, min_cape, min_cin);
    EffSearch s;
    s.init();
    for (int k = 0; k < rd.L; ++k) {
        const double p = rd.P(k);
        if (!eff_valid(p, rd.Tk(k), rd.Td(k))) { put(k, qnan(), qnan()); continue; }
        ParcelResult r;
        eff_lift(rd, k, tb, o, r);
        flags |= r.flags;
        put(k, r.cape, r.cin);
        const bool pass = eff_pass(r.cape, r.cin, min_cape, min_cin);
        if (k == k_mu) gate = pass;
        s.feed(p, pass);
    }
    base_p = gate ? s.base_p : qnan();
    top_p = gate ? s.top_p : qnan();
}

}  // namespace xp
