// hostsim_kinematics.cpp -- TEST-ONLY host build of the storm kinematics column code and the composites
// (xp_kinematics.cuh), the functions storm_kinematics_kernel and composite_parameters_kernel inline, compiled with g++
// so that tests/test_kinematics_hostsim.py can check them against the NumPy restatement on a machine without a GPU.
// Built into tests/hostsim/_build_kinematics by tests/hostsim_kinematics.py; never imported by the product package and
// not a CPU fallback.
#include <algorithm>
#include <cstdint>

#include "../../xarray_parcel_b200/csrc/xp_kinematics.cuh"

// z / u / v [L][n]; su / sv [n]; layers [4][n] (srh bottom, srh top, bwd bottom, bwd top; rows used per flags);
// out [14][n] = right u, right v, left u, left v, mean u, mean v, srh[0..3], srh layer, bwd u, bwd v, bwd magnitude;
// levels_read [n] = 1 + the highest level index the column code read (0: none).
extern "C" void hostsim_storm_kinematics(const double *z, const double *u, const double *v, const double *su,
                                         const double *sv, int64_t n, int L, int motion, int mover, int n_depths,
                                         const double *depths, int srh_layer, int bwd_layer, const double *layers,
                                         double *out, int32_t *levels_read) {
    xp::KinematicsRequest rq;
    rq.motion = motion != 0;
    rq.n_depths = n_depths;
    for (int j = 0; j < xp::kMaxSrhDepths; ++j) rq.depth[j] = j < n_depths ? depths[j] : 0.0;
    rq.srh_layer = srh_layer != 0;
    rq.bwd_layer = bwd_layer != 0;
    rq.mover = (double)mover;
    for (int64_t c = 0; c < n; ++c) {
        int top = 0;
        auto load = [&](int k, double &zz, double &uu, double &vv) {
            top = std::max(top, k + 1);
            zz = z[(int64_t)k * n + c];
            uu = u[(int64_t)k * n + c];
            vv = v[(int64_t)k * n + c];
        };
        xp::KinematicsResult r;
        xp::storm_kinematics(L, load, su[c], sv[c], rq, layers[c], layers[n + c], layers[2 * n + c],
                             layers[3 * n + c], r);
        const double vals[14] = {r.right_u, r.right_v, r.left_u, r.left_v, r.mean_u, r.mean_v, r.srh[0], r.srh[1],
                                 r.srh[2], r.srh[3], r.srh_layer, r.bwd_u, r.bwd_v, r.bwd_magnitude};
        for (int f = 0; f < 14; ++f) out[(int64_t)f * n + c] = vals[f];
        levels_read[c] = top;
    }
}

// in [6][n] = mucape, esrh, ebwd, mlcape, mlcin, lcl height; out [2][n] = scp, stp
extern "C" void hostsim_composites(const double *in, int64_t n, double *out) {
    for (int64_t i = 0; i < n; ++i) {
        out[i] = xp::supercell_composite(in[i], in[n + i], in[2 * n + i]);
        out[n + i] = xp::significant_tornado(in[3 * n + i], in[n + i], in[2 * n + i], in[5 * n + i], in[4 * n + i]);
    }
}
