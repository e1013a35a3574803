// hostsim_effective.cpp -- TEST-ONLY host build of the effective-inflow-layer column code (xp_effective.cuh), the
// functions effective_gate_kernel and effective_layer_kernel inline, compiled with g++ so that
// tests/test_effective_hostsim.py can check them against the NumPy restatement on a machine without a GPU.  Built
// into tests/hostsim/_build_effective by tests/hostsim_effective.py; never imported by the product package and not a
// CPU fallback.
#include <cstdint>

#include "../../xarray_parcel_b200/csrc/xp_effective.cuh"

namespace {

struct HostReader {
    const double *p, *t, *td;
    int64_t ls, pls;
    int L;
    double P(int k) const { return p[(int64_t)k * pls]; }
    double Tk(int k) const { return t[(int64_t)k * ls]; }
    double Td(int k) const { return td[(int64_t)k * ls]; }
};

}  // namespace

// Both modes on every column.  out [5][n] = base, top of the search mode (gate, then eff_search), base, top of the
// all-levels mode, the gate (1 / 0); lcape / lcin [L][n] = the all-levels per-level CAPE / CIN; flags [2] = the flags of each mode.
extern "C" void hostsim_effective(const double *p, int p1d, const double *t, const double *td, int64_t n, int L,
                                  const int *iopts, double mu_depth, double min_cape, double min_cin,
                                  const uint16_t *index_grid, const float *curves, double *out, double *lcape,
                                  double *lcin, uint32_t *flags) {
    xp::Tables tb = {index_grid, curves};
    xp::Opts o;
    o.vtc = iopts[0]; o.log_interp = iopts[1]; o.pos_neg = iopts[2]; o.post_zero = iopts[3];
    o.compat = iopts[4]; o.exact_only = 1; o.vote_mask = 0; o.ml_depth = 100.0; o.mu_depth = mu_depth;
    uint32_t fs = 0, fa = 0;
    for (int64_t c = 0; c < n; ++c) {
        const HostReader rd = {p1d ? p : p + c, t + c, td + c, n, p1d ? 1 : n, L};
        int k_mu;
        double base = xp::qnan(), top = xp::qnan();
        const bool gate = xp::eff_gate(rd, tb, o, min_cape, min_cin, k_mu, fs);
        if (gate) xp::eff_search(rd, tb, o, min_cape, min_cin, k_mu, fs, base, top);
        out[4 * n + c] = gate ? 1.0 : 0.0;
        out[c] = base;
        out[n + c] = top;
        xp::eff_all_levels(rd, tb, o, min_cape, min_cin, fa, out[2 * n + c], out[3 * n + c],
                           [&](int k, double cape, double cin) {
                               lcape[(int64_t)k * n + c] = cape;
                               lcin[(int64_t)k * n + c] = cin;
                           });
    }
    flags[0] = fs;
    flags[1] = fa;
}
