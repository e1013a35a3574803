// xp_downdraft.cu -- downdraft CAPE (xp_downdraft.cuh) as a column kernel.
// One thread per column in a grid-stride loop, float64 arithmetic in the oracle's operation order (no FMA
// contraction); level-major inputs, so each level read of a warp is one coalesced line.  The first pass reads the
// levels up to the first valid one beyond 500 hPa; the second re-reads the levels below the start point, which the
// first pass has just brought into L1 / L2.
#include "xp_kernels.cuh"
#include "xp_downdraft.cuh"

namespace xp {

namespace {

template <typename T>
struct DowndraftParams {
    const T *p, *t, *td;        // [L][N] (p: or shared [L])
    int64_t pls, ls;
    int p1d;
    int L;
    int64_t n;
    int compat;
    Tables tb;
    T *dcape, *p_start, *t_start;   // [N], any may be null
    T *parcel_t;                    // [L][N] with level stride pts, or null
    int64_t pts;
};

template <typename T>
__global__ void __launch_bounds__(128) downdraft_cape_kernel(const __grid_constant__ DowndraftParams<T> prm) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < prm.n; i += (int64_t)gridDim.x * blockDim.x) {
        const T *pc = prm.p1d ? prm.p : prm.p + i;
        auto load = [&](int k, double &p, double &t, double &td) {
            p = (double)pc[(int64_t)k * prm.pls];
            t = (double)prm.t[(int64_t)k * prm.ls + i];
            td = (double)prm.td[(int64_t)k * prm.ls + i];
        };
        DowndraftResult r;
        downdraft_start(prm.L, load, prm.tb, r);
        T *prof = prm.parcel_t ? prm.parcel_t + i : nullptr;
        downdraft_integral(load, prm.tb, prm.compat, r, [&](int k, double v) {
            if (prof) prof[(int64_t)k * prm.pts] = (T)v;
        });
        if (prof)
            for (int k = r.k_end + 1; k < prm.L; ++k) prof[(int64_t)k * prm.pts] = (T)qnan();
        if (prm.dcape) prm.dcape[i] = (T)r.dcape;
        if (prm.p_start) prm.p_start[i] = (T)r.p_start;
        if (prm.t_start) prm.t_start[i] = (T)r.t_start;
    }
}

}  // namespace

template <typename T>
void launch_downdraft_cape(const T *p, int64_t pls, int p1d, const T *t, const T *td, int64_t ls, int L, int64_t n,
                           int compat, const Tables &tb, T *dcape, T *p_start, T *t_start, T *parcel_t, int64_t pts,
                           cudaStream_t stream) {
    if (n <= 0) return;
    DowndraftParams<T> prm;
    prm.p = p; prm.t = t; prm.td = td; prm.pls = pls; prm.ls = ls; prm.p1d = p1d; prm.L = L; prm.n = n;
    prm.compat = compat; prm.tb = tb;
    prm.dcape = dcape; prm.p_start = p_start; prm.t_start = t_start; prm.parcel_t = parcel_t; prm.pts = pts;
    const int64_t blocks = (n + 127) / 128;
    downdraft_cape_kernel<T><<<(unsigned)(blocks < 148 * 64 ? blocks : 148 * 64), 128, 0, stream>>>(prm);
}

#define XP_INST_DOWNDRAFT(T)                                                                                          \
    template void launch_downdraft_cape<T>(const T *, int64_t, int, const T *, const T *, int64_t, int, int64_t, int, \
                                           const Tables &, T *, T *, T *, T *, int64_t, cudaStream_t);
XP_INST_DOWNDRAFT(float)
XP_INST_DOWNDRAFT(double)
#undef XP_INST_DOWNDRAFT

}  // namespace xp
