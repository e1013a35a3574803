// xp_effective.cu -- the effective inflow layer (xp_effective.cuh) in two kernels.
//
// The work per column is uneven: a column whose most-unstable parcel fails the gate costs one lift, a column that
// passes costs one lift per level up to the first failing level above the base (11 lifts on the ERA5 axis, 29 on 70
// model levels, on the synthetic columns).  So
//   effective_gate_kernel   one thread per column: the gate lift; failing columns get their NaN outputs here and the
//                           others are appended to a dense list (one atomicAdd per warp);
//   effective_layer_kernel  a persistent grid over the list; each LANE takes its next column from a global counter
//                           when it has finished the last one, so a long column holds up one lane, not a warp of
//                           columns.  The column's levels are staged in shared memory (every lift re-reads them and
//                           the list's columns are scattered) when that keeps the kernel's occupancy; a shared
//                           pressure axis has its ln p tabulated once per CTA.
// All-levels mode (level CAPE / CIN requested) lists every column with a valid level and lifts every valid level.
// float64 arithmetic, no FMA contraction, as in xp_kernels.cu / xp_list.cu.
#include <type_traits>

#include "xp_kernels_common.cuh"
#include "xp_effective.cuh"

namespace xp {

namespace {

constexpr int kEffColumnBits = 40;              // list entry: column | (most-unstable level << 40)
constexpr uint64_t kEffColumnMask = (1ull << kEffColumnBits) - 1;

template <typename T>
struct EffParams {
    ColsArg<T> cols;
    Tables tb;
    Opts o;
    double min_cape, min_cin;
    int all_levels;
    T *base, *top;                          // [N], either may be null
    T *lcape, *lcin;                        // [L][N] with level stride lls, either may be null
    int64_t lls;
    uint32_t *flags;
    unsigned long long *count;              // [0] list length, [1] next list item of the layer kernel
    uint64_t *list;                         // [N]
};

template <typename T>
__device__ __forceinline__ void eff_store_nan(const EffParams<T> &prm, int64_t col) {
    if (prm.base) prm.base[col] = (T)qnan();
    if (prm.top) prm.top[col] = (T)qnan();
    for (int k = 0; prm.all_levels && k < prm.cols.L; ++k) {
        if (prm.lcape) prm.lcape[(int64_t)k * prm.lls + col] = (T)qnan();
        if (prm.lcin) prm.lcin[(int64_t)k * prm.lls + col] = (T)qnan();
    }
}

template <typename T>
__global__ void __launch_bounds__(128) effective_gate_kernel(const __grid_constant__ EffParams<T> prm) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t w0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x - lane); w0 < prm.cols.n; w0 += stride) {
        // w0 is the same on the 32 lanes of a warp and blockDim.x is a multiple of 32, so the loop condition keeps
        // or drops whole warps: every lane is in the loop here.  Lanes past the last column take part in the ballot.
        const unsigned live = 0xffffffffu;
        const int64_t col = w0 + lane;
        bool push = false;
        uint64_t entry = 0;
        if (col < prm.cols.n) {
            const GlobalReader<T> rd = make_reader(prm.cols, col);
            if (prm.all_levels) {
                for (int k = 0; k < rd.L && !push; ++k) push = eff_valid(rd.P(k), rd.Tk(k), rd.Td(k));
                entry = (uint64_t)col | ((uint64_t)rd.L << kEffColumnBits);
            } else {
                int k_mu;
                uint32_t fl = 0;
                push = eff_gate(rd, prm.tb, prm.o, prm.min_cape, prm.min_cin, k_mu, fl);
                if (fl && prm.flags) atomicOr(prm.flags, fl);
                entry = (uint64_t)col | ((uint64_t)k_mu << kEffColumnBits);
            }
            if (!push) eff_store_nan(prm, col);
        }
        const unsigned m = __ballot_sync(live, push);
        if (m) {
            const int leader = __ffs(m) - 1;
            unsigned long long at = 0;
            if (lane == leader) at = atomicAdd(prm.count, (unsigned long long)__popc(m));
            at = __shfl_sync(live, at, leader);
            if (push) {
                const unsigned long long i = at + __popc(m & ((1u << lane) - 1u));
                XP_CHECK((int64_t)i < prm.cols.n);
                prm.list[i] = entry;
            }
        }
    }
}

// Column reader of the layer kernel.  STAGED: T and Td (and, with STAGE_P, p) come from this thread's slots in
// shared memory, s[(f * L + k) * nt] for field f = 0 T, 1 Td, 2 p -- the same values GlobalReader loads, converted
// the same way, so the column code gets the same bits.
template <typename T, bool STAGE_P, bool STAGED>
struct EffReader {
    GlobalReader<T> g;
    const T *s;
    int nt, L;
    __device__ __forceinline__ double P(int k) const {
        if constexpr (STAGE_P) return (double)s[(2 * L + k) * nt];
        else return g.P(k);
    }
    __device__ __forceinline__ double Tk(int k) const {
        if constexpr (STAGED) return (double)s[k * nt];
        else return g.Tk(k);
    }
    __device__ __forceinline__ double Td(int k) const {
        if constexpr (STAGED) return (double)s[(L + k) * nt];
        else return g.Td(k);
    }
};

// A shared pressure axis: ln p of its levels tabulated per CTA by the same log() the column code would call.
template <typename T, bool STAGED>
struct EffAxisReader : EffReader<T, false, STAGED> {
    const double *ln_axis;
    __device__ __forceinline__ double LnP(int k) const { return ln_axis[k]; }
};

template <typename T, bool AXIS, bool STAGED>
__global__ void __launch_bounds__(128) effective_layer_kernel(const __grid_constant__ EffParams<T> prm) {
    extern __shared__ __align__(8) unsigned char eff_smem[];
    const int L = prm.cols.L, nt = (int)blockDim.x;
    double *s_ln = reinterpret_cast<double *>(eff_smem);
    T *s_slots = reinterpret_cast<T *>(eff_smem + (AXIS ? (size_t)L * sizeof(double) : 0)) + threadIdx.x;
    if constexpr (AXIS) {
        for (int k = threadIdx.x; k < L; k += blockDim.x)
            s_ln[k] = xp_log((double)__ldg(prm.cols.p + (int64_t)k * prm.cols.pls));
        __syncthreads();
    }
    using Reader = std::conditional_t<AXIS, EffAxisReader<T, STAGED>, EffReader<T, STAGED, STAGED>>;
    const unsigned long long total = *(volatile const unsigned long long *)prm.count;
    for (;;) {
        const unsigned long long it = atomicAdd(prm.count + 1, 1ull);
        if (it >= total) break;
        const uint64_t e = prm.list[it];
        const int64_t col = (int64_t)(e & kEffColumnMask);
        const int k_known = (int)(e >> kEffColumnBits);
        XP_CHECK(col < prm.cols.n && k_known <= L);
        Reader rd;
        rd.g = make_reader(prm.cols, col);
        rd.s = s_slots;
        rd.nt = nt;
        rd.L = L;
        if constexpr (AXIS) rd.ln_axis = s_ln;
        if constexpr (STAGED) {
            // only this thread reads its slots back: no barrier
            for (int k = 0; k < L; ++k) {
                s_slots[k * nt] = __ldg(rd.g.t + (int64_t)k * rd.g.ls);
                s_slots[(L + k) * nt] = __ldg(rd.g.td + (int64_t)k * rd.g.ls);
                if constexpr (!AXIS) s_slots[(2 * L + k) * nt] = __ldg(rd.g.p + (int64_t)k * rd.g.pls);
            }
        }
        uint32_t fl = 0;
        double base_p, top_p;
        if (prm.all_levels) {
            T *lc = prm.lcape ? prm.lcape + col : nullptr;
            T *ln = prm.lcin ? prm.lcin + col : nullptr;
            eff_all_levels(rd, prm.tb, prm.o, prm.min_cape, prm.min_cin, fl, base_p, top_p,
                           [&](int k, double cape, double cin) {
                               if (lc) lc[(int64_t)k * prm.lls] = (T)cape;
                               if (ln) ln[(int64_t)k * prm.lls] = (T)cin;
                           });
        } else {
            eff_search(rd, prm.tb, prm.o, prm.min_cape, prm.min_cin, k_known, fl, base_p, top_p);
        }
        if (prm.base) prm.base[col] = (T)base_p;
        if (prm.top) prm.top[col] = (T)top_p;
        if (fl && prm.flags) atomicOr(prm.flags, fl);
    }
}

// Stage the columns when the staged kernel keeps the occupancy of the unstaged one (at 37 float levels a thread's
// T / Td slots are 296 bytes; at 70 per-column float64 levels 1.7 KB, which would cost resident warps).
template <typename T, bool AXIS>
int launch_layer(const EffParams<T> &prm, int sm_count, cudaStream_t stream) {
    const int L = prm.cols.L;
    const size_t ln_bytes = AXIS ? (size_t)L * sizeof(double) : 0;
    const size_t staged_bytes = ln_bytes + (size_t)(AXIS ? 2 : 3) * L * 128 * sizeof(T);
    auto k_plain = effective_layer_kernel<T, AXIS, false>;
    auto k_staged = effective_layer_kernel<T, AXIS, true>;
    int dev = 0, optin = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if constexpr (AXIS) {
        if (ln_bytes > (size_t)optin) return -1;
    }
    // per device, so set on every launch (a host-side call of about a microsecond)
    if (cudaFuncSetAttribute(k_plain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ln_bytes) != cudaSuccess) return -1;
    int occ_plain = 0, occ_staged = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_plain, k_plain, 128, ln_bytes);
    if (staged_bytes <= (size_t)optin &&
        cudaFuncSetAttribute(k_staged, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged_bytes) == cudaSuccess)
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_staged, k_staged, 128, staged_bytes);
    cudaGetLastError();     // an occupancy query that failed leaves its count at 0; do not report it as the launch's
    if (occ_staged > 0 && occ_staged >= occ_plain)
        k_staged<<<sm_count * occ_staged, 128, staged_bytes, stream>>>(prm);
    else
        k_plain<<<sm_count * (occ_plain > 0 ? occ_plain : 1), 128, ln_bytes, stream>>>(prm);
    return 0;
}

}  // namespace

size_t effective_scratch_bytes(int64_t n) { return 2 * sizeof(unsigned long long) + (size_t)n * sizeof(uint64_t); }

template <typename T>
int launch_effective(const ColsArg<T> &cols, const Tables &tb, const Opts &o, double min_cape, double min_cin,
                     T *base, T *top, T *lcape, T *lcin, int64_t lls, uint32_t *flags, void *scratch, int sm_count,
                     cudaStream_t stream) {
    if (cols.n <= 0) return 0;
    EffParams<T> prm;
    prm.cols = cols; prm.tb = tb; prm.o = o; prm.min_cape = min_cape; prm.min_cin = min_cin;
    prm.all_levels = (lcape || lcin) ? 1 : 0;
    prm.base = base; prm.top = top; prm.lcape = lcape; prm.lcin = lcin; prm.lls = lls;
    prm.flags = flags;
    prm.count = static_cast<unsigned long long *>(scratch);
    prm.list = reinterpret_cast<uint64_t *>(prm.count + 2);
    cudaMemsetAsync(prm.count, 0, 2 * sizeof(unsigned long long), stream);
    const int64_t blocks = (cols.n + 127) / 128;
    effective_gate_kernel<T><<<(unsigned)(blocks < sm_count * 64 ? blocks : sm_count * 64), 128, 0, stream>>>(prm);
    return cols.p1d ? launch_layer<T, true>(prm, sm_count, stream) : launch_layer<T, false>(prm, sm_count, stream);
}

#define XP_INST_EFFECTIVE(T)                                                                                        \
    template int launch_effective<T>(const ColsArg<T> &, const Tables &, const Opts &, double, double, T *, T *, \
                                     T *, T *, int64_t, uint32_t *, void *, int, cudaStream_t);
XP_INST_EFFECTIVE(float)
XP_INST_EFFECTIVE(double)
#undef XP_INST_EFFECTIVE

}  // namespace xp
