// xp_kinematics.cu -- storm kinematics (xp_kinematics.cuh) as a column kernel, and the supercell / tornado composites
// as a pointwise kernel.  float64 arithmetic in the order of xp_kinematics.cuh (no FMA contraction).
// storm_kinematics_kernel: one thread per column in a grid-stride loop; level-major inputs, so each level read of a
// warp is one coalesced line per field; a thread stops reading at the first profile point at or above the highest
// bound its column needs.  No shared memory and no warp collectives.
#include "xp_kernels.cuh"
#include "xp_kinematics.cuh"

namespace xp {

namespace {

template <typename T>
struct KinematicsParams {
    const T *z, *u, *v;             // [L][N], level stride ls
    const T *su, *sv;               // [N]
    const T *sb, *st, *bb, *bt;     // [N] or null
    int64_t ls, n;
    int L;
    KinematicsRequest rq;
    T *right_u, *right_v, *left_u, *left_v, *mean_u, *mean_v;   // [N], any may be null
    T *srh[kMaxSrhDepths];
    T *srh_layer, *bwd_u, *bwd_v, *bwd_mag;
};

template <typename T>
__device__ __forceinline__ void put(T *out, int64_t i, double x) {
    if (out) out[i] = (T)x;
}

template <typename T>
__global__ void __launch_bounds__(128) storm_kinematics_kernel(const __grid_constant__ KinematicsParams<T> prm) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < prm.n; i += (int64_t)gridDim.x * blockDim.x) {
        auto load = [&](int k, double &z, double &u, double &v) {
            const int64_t o = (int64_t)k * prm.ls + i;
            z = (double)prm.z[o];
            u = (double)prm.u[o];
            v = (double)prm.v[o];
        };
        const double nan = qnan();
        KinematicsResult r;
        storm_kinematics(prm.L, load, (double)prm.su[i], (double)prm.sv[i], prm.rq,
                         prm.sb ? (double)prm.sb[i] : nan, prm.st ? (double)prm.st[i] : nan,
                         prm.bb ? (double)prm.bb[i] : nan, prm.bt ? (double)prm.bt[i] : nan, r);
        put(prm.right_u, i, r.right_u);
        put(prm.right_v, i, r.right_v);
        put(prm.left_u, i, r.left_u);
        put(prm.left_v, i, r.left_v);
        put(prm.mean_u, i, r.mean_u);
        put(prm.mean_v, i, r.mean_v);
#pragma unroll
        for (int j = 0; j < kMaxSrhDepths; ++j) put(prm.srh[j], i, r.srh[j]);
        put(prm.srh_layer, i, r.srh_layer);
        put(prm.bwd_u, i, r.bwd_u);
        put(prm.bwd_v, i, r.bwd_v);
        put(prm.bwd_mag, i, r.bwd_magnitude);
    }
}

template <typename T>
__global__ void __launch_bounds__(256) composite_parameters_kernel(const T *mucape, const T *esrh, const T *ebwd,
                                                                   const T *mlcape, const T *mlcin, const T *lcl_h,
                                                                   int64_t n, T *scp, T *stp) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double s = (double)esrh[i], b = (double)ebwd[i];
        if (scp) scp[i] = (T)supercell_composite((double)mucape[i], s, b);
        if (stp) stp[i] = (T)significant_tornado((double)mlcape[i], s, b, (double)lcl_h[i], (double)mlcin[i]);
    }
}

unsigned grid_for(int64_t n, int threads) {
    const int64_t blocks = (n + threads - 1) / threads;
    return (unsigned)(blocks < 148 * 64 ? blocks : 148 * 64);
}

}  // namespace

template <typename T>
void launch_storm_kinematics(const T *z, const T *u, const T *v, const T *su, const T *sv, int64_t ls, int L,
                             int64_t n, const KinematicsRequest &rq, const T *sb, const T *st, const T *bb,
                             const T *bt, T *const *motion6, T *const *srh4, T *srh_layer, T *const *bwd3,
                             cudaStream_t stream) {
    if (n <= 0) return;
    KinematicsParams<T> prm;
    prm.z = z; prm.u = u; prm.v = v; prm.su = su; prm.sv = sv;
    prm.sb = sb; prm.st = st; prm.bb = bb; prm.bt = bt;
    prm.ls = ls; prm.n = n; prm.L = L; prm.rq = rq;
    prm.right_u = motion6[0]; prm.right_v = motion6[1]; prm.left_u = motion6[2]; prm.left_v = motion6[3];
    prm.mean_u = motion6[4]; prm.mean_v = motion6[5];
    for (int j = 0; j < kMaxSrhDepths; ++j) prm.srh[j] = srh4[j];
    prm.srh_layer = srh_layer;
    prm.bwd_u = bwd3[0]; prm.bwd_v = bwd3[1]; prm.bwd_mag = bwd3[2];
    storm_kinematics_kernel<T><<<grid_for(n, 128), 128, 0, stream>>>(prm);
}

template <typename T>
void launch_composite_parameters(const T *mucape, const T *esrh, const T *ebwd, const T *mlcape, const T *mlcin,
                                 const T *lcl_h, int64_t n, T *scp, T *stp, cudaStream_t stream) {
    if (n <= 0) return;
    composite_parameters_kernel<T><<<grid_for(n, 256), 256, 0, stream>>>(mucape, esrh, ebwd, mlcape, mlcin, lcl_h, n,
                                                                          scp, stp);
}

#define XP_INST_KINEMATICS(T)                                                                                         \
    template void launch_storm_kinematics<T>(const T *, const T *, const T *, const T *, const T *, int64_t, int,     \
                                             int64_t, const KinematicsRequest &, const T *, const T *, const T *,     \
                                             const T *, T *const *, T *const *, T *, T *const *, cudaStream_t);       \
    template void launch_composite_parameters<T>(const T *, const T *, const T *, const T *, const T *, const T *,    \
                                                 int64_t, T *, T *, cudaStream_t);
XP_INST_KINEMATICS(float)
XP_INST_KINEMATICS(double)
#undef XP_INST_KINEMATICS

}  // namespace xp
