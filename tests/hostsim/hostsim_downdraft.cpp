// hostsim_downdraft.cpp -- TEST-ONLY host build of the downdraft CAPE column code (xp_downdraft.cuh), the functions
// downdraft_cape_kernel inlines, compiled with g++ so that tests/test_downdraft_hostsim.py can check them against the
// NumPy restatement on a machine without a GPU.  Built into tests/hostsim/_build_downdraft by
// tests/hostsim_downdraft.py; never imported by the product package and not a CPU fallback.
#include <algorithm>
#include <cstdint>

#include "../../xarray_parcel_b200/csrc/xp_downdraft.cuh"

// out [3][n] = dcape, start pressure, start temperature; prof [L][n] (or null) = the parcel temperature;
// levels_read [n] (or null) = 1 + the highest level index the column code read.
extern "C" void hostsim_downdraft_cape(const double *p, int p1d, const double *t, const double *td, int64_t n, int L,
                                       int compat, const uint16_t *index_grid, const float *curves,
                                       double *out /*[3][n]*/, double *prof /*[L][n]*/, int32_t *levels_read) {
    xp::Tables tb = {index_grid, curves};
    for (int64_t c = 0; c < n; ++c) {
        const double *pc = p1d ? p : p + c;
        const int64_t pls = p1d ? 1 : n;
        int top = 0;
        auto load = [&](int k, double &pp, double &tt, double &dd) {
            top = std::max(top, k + 1);
            pp = pc[(int64_t)k * pls];
            tt = t[(int64_t)k * n + c];
            dd = td[(int64_t)k * n + c];
        };
        xp::DowndraftResult r;
        xp::downdraft_start(L, load, tb, r);
        auto put = [&](int k, double v) { if (prof) prof[(int64_t)k * n + c] = v; };
        xp::downdraft_integral(load, tb, compat, r, put);
        if (prof)
            for (int k = r.k_end + 1; k < L; ++k) prof[(int64_t)k * n + c] = xp::qnan();
        out[c] = r.dcape;
        out[n + c] = r.p_start;
        out[2 * n + c] = r.t_start;
        if (levels_read) levels_read[c] = top;
    }
}
