// xp_fast.cu -- sm_100a kernels of the float32 fast path (see xp_fast.cuh) and of the exact-path
// fix-up over the compact list of columns whose decisions were uncertain in float32.
#include <algorithm>
#include <cstdlib>

#include "xp_fast.cuh"
#include "xp_fast_pcol.cuh"
#include "xp_fast6.cuh"
#include "xp_fast7.cuh"
#include "xp_fast_pcol6.cuh"
#include "xp_fast_pcol7.cuh"
#include "xp_kernels.cuh"

// Streaming read of column data (each element is used once): evict-first in L2 so that it does not push the
// moist-adiabat tables (gathered many times) out.  XP_STREAM_LOADS=0 at build time restores plain loads.
#ifndef XP_STREAM_LOADS
#define XP_STREAM_LOADS 1
#endif
#if XP_STREAM_LOADS
#define XP_LDSTREAM(ptr) __ldcs(ptr)
#else
#define XP_LDSTREAM(ptr) __ldg(ptr)
#endif

namespace xp {

using fast::Coef;
using fast::Prep;

namespace {

// ---- prep kernels: axis constants (one thread) and the cubic coefficient table -----------------------
template <typename TP>
__global__ void fast_prep_kernel(const TP *__restrict__ p, int64_t pls, int L, Opts o, Prep *out) {
    if (threadIdx.x < L && threadIdx.x < fast::kMaxLevels) fast::compute_prep_level(p, pls, threadIdx.x, *out);
    __syncthreads();
    if (threadIdx.x == 0) fast::compute_prep_axis(L, o, *out);
}

// tv = 1: cubics of the saturated parcel's VIRTUAL temperature (v6 sweep, xp_fast6.cuh); 0: of its temperature
__global__ void fast_coef_kernel(const Prep *__restrict__ prep, const float *__restrict__ curves, Coef *__restrict__ coef,
                                 int tv) {
    const int k = blockIdx.x, m = threadIdx.x;
    if (!prep->ok || k >= prep->n_table || m >= fast::kNI) return;
    coef[(size_t)k * fast::kNI + m] = tv ? fast::compute_coef_tv(*prep, curves, k, m) : fast::compute_coef(*prep, curves, k, m);
}

// ---- the fast suite kernel ---------------------------------------------------------------------------------------
template <typename T>
struct FastParamsT {
    const T *t, *td;
    int64_t n, ls;
    const Prep *prep;
    const Coef *coef;
    Tables tb;
    Opts o;
    unsigned kinds;
    OutArg<T> outs[3];
    uint32_t *list;          // 3 regions of n entries (see ListParams)
    uint32_t *list_count;
    int stash_levels;        // levels of T/Td per thread that fit in shared memory after the table (v6 sweep)
    int dense_out;           // the requested outputs are exactly the 9 scalars per kind + parcel p/T/Td of ML, MU
};
using FastParams = FastParamsT<float>;

struct GlobalRd {
    const float *t, *td;
    int64_t ls;
    __device__ __forceinline__ float T(int k) const { return __ldg(t + (int64_t)k * ls); }
    __device__ __forceinline__ float Td(int k) const { return __ldg(td + (int64_t)k * ls); }
    __device__ __forceinline__ const float *tptr(int k) const { return t + (int64_t)k * ls; }
    __device__ __forceinline__ const float *tdptr(int k) const { return td + (int64_t)k * ls; }
    __device__ __forceinline__ int64_t stride() const { return ls; }
    static __device__ __forceinline__ float ld(const float *p) { return __ldg(p); }
    static __device__ __forceinline__ void prefetch(const float *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
};

// v6 sweep: 32-bit element offsets from the array bases (see Sweep6 in xp_fast6.cuh)
// T = double: float64 columns.  The sweep consumes them rounded to float32; the parcel levels are re-read in float64
// (ldT64 / ldTd64) by suite_column7.
template <typename T>
struct GlobalRd32T {
    static constexpr bool kDouble = sizeof(T) == 8;
    const T *t, *td;
    uint32_t col, lstride;
    uint64_t limit;                       // elements addressable from the bases (XP_BOUNDS_CHECK builds only)
    __device__ __forceinline__ uint32_t off0() const { return col; }
    __device__ __forceinline__ uint32_t ls() const { return lstride; }
    __device__ __forceinline__ float ldT(uint32_t off) const { XP_CHECK(off < limit); return (float)__ldg(t + off); }
    __device__ __forceinline__ float ldTd(uint32_t off) const { XP_CHECK(off < limit); return (float)__ldg(td + off); }
    __device__ __forceinline__ double ldT64(uint32_t off) const { XP_CHECK(off < limit); return (double)__ldg(t + off); }
    __device__ __forceinline__ double ldTd64(uint32_t off) const { XP_CHECK(off < limit); return (double)__ldg(td + off); }
    __device__ __forceinline__ void prefetch(uint32_t off) const {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(t + off));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(td + off));
    }
};
using GlobalRd32 = GlobalRd32T<float>;

struct SmemCoefRow {
    const Coef *row;
#ifdef XP_BOUNDS_CHECK
    const Coef *lo, *hi;                  // the table in shared memory
#endif
    __device__ __forceinline__ void advance() { row += fast::kNI; }
    __device__ __forceinline__ Coef at(int m) const {
#ifdef XP_BOUNDS_CHECK
        XP_CHECK(m >= 0 && m < fast::kNI && row + m >= lo && row + m < hi);
#endif
        const float4 v = *reinterpret_cast<const float4 *>(row + m);
        return Coef{v.x, v.y, v.z, v.w};
    }
};
struct SmemCoef {
    const Coef *base;
    int rows;                             // levels held
    __device__ __forceinline__ SmemCoefRow row(int k) const {
#ifdef XP_BOUNDS_CHECK
        return SmemCoefRow{base + k * fast::kNI, base, base + (size_t)rows * fast::kNI};
#else
        return SmemCoefRow{base + k * fast::kNI};
#endif
    }
};

template <typename T>
__device__ __forceinline__ void store_fast(const OutArg<T> &o, int64_t col, const fast::FResult &r) {
    if (o.cape) o.cape[col] = (T)r.cape;
    if (o.cin) o.cin[col] = (T)r.cin;
    if (o.lcl_p) o.lcl_p[col] = (T)r.lcl_p;
    if (o.lcl_t) o.lcl_t[col] = (T)r.lcl_t;
    if (o.lcl_tv) o.lcl_tv[col] = (T)r.lcl_tv;
    if (o.lfc_p) o.lfc_p[col] = (T)r.lfc_p;
    if (o.lfc_t) o.lfc_t[col] = (T)r.lfc_t;
    if (o.el_p) o.el_p[col] = (T)r.el_p;
    if (o.el_t) o.el_t[col] = (T)r.el_t;
    if (o.par_p) o.par_p[col] = (T)r.par_p;
    if (o.par_t) o.par_t[col] = (T)r.par_t;
    if (o.par_td) o.par_td[col] = (T)r.par_td;
    if (o.shift) o.shift[col] = r.shift;
}

// Every scalar output of the kind is requested (the usual case): no pointer checks.
template <typename T>
__device__ __forceinline__ void store_fast_all(const OutArg<T> &o, int64_t col, const fast::FResult &r, bool parcel) {
    o.cape[col] = (T)r.cape; o.cin[col] = (T)r.cin;
    o.lcl_p[col] = (T)r.lcl_p; o.lcl_t[col] = (T)r.lcl_t; o.lcl_tv[col] = (T)r.lcl_tv;
    o.lfc_p[col] = (T)r.lfc_p; o.lfc_t[col] = (T)r.lfc_t; o.el_p[col] = (T)r.el_p; o.el_t[col] = (T)r.el_t;
    if (parcel) { o.par_p[col] = (T)r.par_p; o.par_t[col] = (T)r.par_t; o.par_td[col] = (T)r.par_td; }
}

#ifndef XP_FAST_THREADS
#define XP_FAST_THREADS 640
#endif
constexpr int kFastThreads = XP_FAST_THREADS;   // threads of the one persistent CTA per SM

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Per-thread column of the environment curve in shared memory: element (level k, thread t) at
// base[k * blockDim.x + t] -- consecutive threads hit consecutive banks.
struct EnvSmem {
    static constexpr bool kStaged = true, kFullPass = true;
    float *base;
    int stride;
    __device__ __forceinline__ void put(int k, float v) { base[k * stride] = v; }
    __device__ __forceinline__ float get(int k) const { return base[k * stride]; }
};

// T/Td of the lowest levels of every thread's column: element (level k, T|Td, thread) at
// base[(2 k + which) * blockDim.x + thread] -- conflict-free.
struct StashSmem {
    float *base;
    int stride, cap;
    __device__ __forceinline__ int capacity() const { return cap; }
    __device__ __forceinline__ void put(int k, float t, float td) {
        XP_CHECK(k >= 0 && k < cap);
        base[(2 * k) * stride] = t; base[(2 * k + 1) * stride] = td;
    }
    __device__ __forceinline__ void get(int k, float &t, float &td) const {
        XP_CHECK(k >= 0 && k < cap);
        t = base[(2 * k) * stride]; td = base[(2 * k + 1) * stride];
    }
};

// STAGED: 0 = environment recomputed in the sweep (default options: the v6 sweep of xp_fast6.cuh); 1 = environment
// curve staged in shared memory + early termination; 2 = recomputed, with a first pass over all levels for the
// early-termination bound; 3 = the v7 sweep of xp_fast7.cuh (default options only; shared memory as 0); 4 = the v7 sweep
// with specific humidity in place of the dewpoint, converted in the load stage (xp_columns.dewpoint_is_specific_humidity).
// T: element type of the columns and of the outputs (double only with the v7 sweep, STAGED 3).
template <unsigned KINDS, int MODE, int THREADS, int STAGED, typename T = float>
__global__ void __launch_bounds__(THREADS, 1) suite_fast_kernel(const __grid_constant__ FastParamsT<T> prm) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t mbar;
    Prep *s_prep = reinterpret_cast<Prep *>(smem_raw);
    constexpr size_t kPrepBytes = (sizeof(Prep) + 127) & ~(size_t)127;
    Coef *s_coef = reinterpret_cast<Coef *>(smem_raw + kPrepBytes);

    // Prep (a few KB): plain cooperative copy
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(prm.prep);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_prep);
        for (int i = threadIdx.x; i < (int)(sizeof(Prep) / 4); i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const Prep &pr = *s_prep;
    if (!pr.ok) {
        // the axis does not qualify: every column goes to the exact path
        for (int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; col < prm.n;
             col += (int64_t)gridDim.x * blockDim.x) {
            push_redo(prm.list, prm.list_count, prm.n, col, prm.kinds);
        }
        return;
    }
    // the adiabat table: one bulk asynchronous copy (TMA) per level row into shared memory
    const uint32_t row_bytes = fast::kNI * sizeof(Coef);
    if (threadIdx.x == 0) {
        const uint32_t total = row_bytes * (uint32_t)pr.n_table;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(total) : "memory");
        for (int k = 0; k < pr.n_table; ++k) {
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                    smem_u32(s_coef + (size_t)k * fast::kNI)),
                "l"(prm.coef + (size_t)k * fast::kNI), "r"(row_bytes), "r"(smem_u32(&mbar))
                : "memory");
        }
    }
    {   // everyone waits for the table (phase 0)
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done) : "r"(smem_u32(&mbar)), "r"(0u) : "memory");
        }
    }
    const SmemCoef cf{s_coef, pr.n_table};
    float *s_env = reinterpret_cast<float *>(s_coef + (size_t)pr.n_table * fast::kNI);
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < prm.n; base += (int64_t)gridDim.x * blockDim.x) {
        // lanes past the end redo the last column (warp-uniform votes need every lane) and do not store
        const bool valid = base + threadIdx.x < prm.n;
        const int64_t col = valid ? base + threadIdx.x : prm.n - 1;
        fast::FResult res[3];
        unsigned redo;
        if constexpr (MODE == 1 && (STAGED == 3 || STAGED == 4)) {
            StashSmem st{s_env + threadIdx.x, (int)blockDim.x, prm.stash_levels};
            const GlobalRd32T<T> rd32{prm.t, prm.td, (uint32_t)col, (uint32_t)prm.ls, (uint64_t)prm.n + (uint64_t)(pr.L - 1) * (uint64_t)prm.ls};
            redo = fast::suite_column7<KINDS, STAGED == 4>(rd32, cf, pr, prm.tb, prm.o, st, res);
        } else if constexpr (MODE == 1 && STAGED == 0) {
            // default options: the v6 sweep on the virtual-temperature table (xp_fast6.cuh); the shared
            // memory left after the table stashes T/Td of the lowest levels of every thread's column
            StashSmem st{s_env + threadIdx.x, (int)blockDim.x, prm.stash_levels};
            const GlobalRd32 rd32{prm.t, prm.td, (uint32_t)col, (uint32_t)prm.ls, (uint64_t)prm.n + (uint64_t)(pr.L - 1) * (uint64_t)prm.ls};
            redo = fast::suite_column6<KINDS>(rd32, cf, pr, prm.tb, prm.o, st, res);
        } else if constexpr (STAGED == 1) {
            const GlobalRd rd{prm.t + col, prm.td + col, prm.ls};
            EnvSmem env{s_env + threadIdx.x, (int)blockDim.x};
            redo = fast::suite_column<KINDS, MODE>(rd, cf, pr, prm.tb, prm.o, env, res);
        } else if constexpr (STAGED == 2) {
            const GlobalRd rd{prm.t + col, prm.td + col, prm.ls};
            fast::EnvMinOnly env;
            redo = fast::suite_column<KINDS, MODE>(rd, cf, pr, prm.tb, prm.o, env, res);
        } else {
            const GlobalRd rd{prm.t + col, prm.td + col, prm.ls};
            fast::EnvRecompute env;
            redo = fast::suite_column<KINDS, MODE>(rd, cf, pr, prm.tb, prm.o, env, res);
        }
        if (!valid) continue;
        if (prm.dense_out) {
            // cape .. el_temperature of every kind, parcel p/T/Td of ML and MU, nothing else
            if (KINDS & 1u) store_fast_all(prm.outs[0], col, res[0], false);
            if (KINDS & 2u) store_fast_all(prm.outs[1], col, res[1], true);
            if (KINDS & 4u) store_fast_all(prm.outs[2], col, res[2], true);
        } else {
            if (KINDS & 1u) store_fast(prm.outs[0], col, res[0]);
            if (KINDS & 2u) store_fast(prm.outs[1], col, res[1]);
            if (KINDS & 4u) store_fast(prm.outs[2], col, res[2]);
        }
        if (redo) push_redo(prm.list, prm.list_count, prm.n, col, redo);
    }
}

// ---- the fast suite kernel for per-column pressure (xp_fast_pcol.cuh) ------------------------------------------
struct PColRd {
    const float *p, *t, *td;
    int64_t ls, pls;
    __device__ __forceinline__ float P(int k) const { return __ldg(p + (int64_t)k * pls); }
    __device__ __forceinline__ float T(int k) const { return __ldg(t + (int64_t)k * ls); }
    __device__ __forceinline__ float Td(int k) const { return __ldg(td + (int64_t)k * ls); }
    __device__ __forceinline__ const float *pptr(int k) const { return p + (int64_t)k * pls; }
    __device__ __forceinline__ const float *tptr(int k) const { return t + (int64_t)k * ls; }
    __device__ __forceinline__ const float *tdptr(int k) const { return td + (int64_t)k * ls; }
    __device__ __forceinline__ int64_t stride() const { return ls; }
    __device__ __forceinline__ int64_t pstride() const { return pls; }
    static __device__ __forceinline__ float ld(const float *q) { return __ldg(q); }
};

struct PColParams {
    const float *p, *t, *td;
    int64_t n, ls, pls;
    int L;
    Tables tb;
    Opts o;
    OutArg<float> outs[3];
    uint32_t *list;
    uint32_t *list_count;
};

#ifndef XP_PCOL_THREADS
#define XP_PCOL_THREADS 256
#endif
constexpr int kPColThreads = XP_PCOL_THREADS;
// CTAs per SM the per-column-pressure kernel is compiled for: a single parcel kind without profile rows fits 85
// registers (three 256-thread CTAs: measured 1.09 vs 0.95 G columns/s on 1 M x 70 surface-based); two or three kinds
// spill there (SB+ML: 0.48 vs 0.70 G) and stay at two CTAs x 128 registers.
constexpr int pcol_ctas(unsigned kinds, bool profile) {
    return (!profile && (kinds == 1u || kinds == 2u || kinds == 4u)) ? 3 : 2;
}

// parcel_profile_with_lcl rows (PF:806-931) of the fast path: [L+1][N] arrays per kind, NULL = not wanted
struct ProfileWriter {
    static constexpr bool kEnabled = true;
    const OutArg<float> *outs;
    int64_t col;
    int L;
    __device__ __forceinline__ void put(int q, int row, float p, float tp, float tv, float et, float etv,
                                        float etd) const {
        if ((unsigned)row > (unsigned)L) return;          // rows 0..L exist
        const OutArg<float> &o = outs[q];
        const int64_t off = (int64_t)row * o.prof_ls + col;
        if (o.prof_p) o.prof_p[off] = p;
        if (o.prof_t) o.prof_t[off] = tp;
        if (o.prof_tv) o.prof_tv[off] = tv;
        if (o.prof_et) o.prof_et[off] = et;
        if (o.prof_etv) o.prof_etv[off] = etv;
        if (o.prof_etd) o.prof_etd[off] = etd;
    }
};

// Per-thread ring of (p, T, Td) levels in dynamic shared memory for the re-based profile sweep (fast::NoRing in
// xp_fast_pcol.cuh): element (slot, which, thread) at base[(3 slot + which) * blockDim.x + thread] -- conflict-free.
constexpr int kPColRingLevels = 48;        // covers a most-unstable search over 43 levels (300 hPa of a 90-level grid)
constexpr int kPColRingThreads = 128;      // 48 x 3 x 4 B x 128 = 72 KB per CTA: three CTAs per SM
struct RingSmem {
    static constexpr bool kEnabled = true;
    float *base;
    int stride;
    __device__ __forceinline__ int capacity() const { return kPColRingLevels; }
    __device__ __forceinline__ void put(int s, float p, float t, float td) {
        XP_CHECK(s >= 0 && s < kPColRingLevels);
        base[(3 * s) * stride] = p; base[(3 * s + 1) * stride] = t; base[(3 * s + 2) * stride] = td;
    }
    __device__ __forceinline__ void get(int s, float &p, float &t, float &td) const {
        XP_CHECK(s >= 0 && s < kPColRingLevels);
        p = base[(3 * s) * stride]; t = base[(3 * s + 1) * stride]; td = base[(3 * s + 2) * stride];
    }
};

// RING: one lifted kind with profile rows -- the re-based sweep reads its levels through the shared-memory ring
// (kPColRingThreads threads per CTA); everything else reads directly (kPColThreads).
template <unsigned KINDS, int MODE, bool PROFILE, bool QIN = false, bool RING = false>
__global__ void __launch_bounds__(RING ? kPColRingThreads : kPColThreads, RING ? 3 : pcol_ctas(KINDS, PROFILE))
suite_fast_pcol_kernel(const __grid_constant__ PColParams prm) {
    extern __shared__ __align__(16) float s_ring[];
    const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= prm.n) return;
    const PColRd rd{prm.p + col, prm.t + col, prm.td + col, prm.ls, prm.pls};
    fast::FResult res[3];
    unsigned redo;
    if constexpr (PROFILE && RING) {
        ProfileWriter pw{prm.outs, col, prm.L};
        RingSmem ring{s_ring + threadIdx.x, (int)blockDim.x};
        redo = fast::suite_column_pcol<KINDS, MODE, QIN>(rd, prm.L, prm.tb, prm.o, pw, ring, fast::NoPTab(), res);
    } else if constexpr (PROFILE) {
        ProfileWriter pw{prm.outs, col, prm.L};
        fast::NoRing ring;
        redo = fast::suite_column_pcol<KINDS, MODE, QIN>(rd, prm.L, prm.tb, prm.o, pw, ring, fast::NoPTab(), res);
    } else {
        fast::NoProfile np;
        fast::NoRing ring;
        redo = fast::suite_column_pcol<KINDS, MODE, QIN>(rd, prm.L, prm.tb, prm.o, np, ring, fast::NoPTab(), res);
    }
    if (KINDS & 1u) store_fast(prm.outs[0], col, res[0]);
    if (KINDS & 2u) store_fast(prm.outs[1], col, res[1]);
    if (KINDS & 4u) store_fast(prm.outs[2], col, res[2]);
    if (redo) push_redo(prm.list, prm.list_count, prm.n, col, redo);
}

// ---- per-column pressure with the adiabat family in SHARED memory (fast::PTabView, xp_fast_pcol.cuh) ----------------
// Default options, scalar outputs.  Persistent: one 512-thread CTA per SM stages the 136 KB table once, by bulk
// asynchronous copies (TMA, one per node row) completing on an mbarrier, then walks over 512-column tiles.
__global__ void ptab_coef_kernel(const float *__restrict__ curves, Coef *__restrict__ coef) {
    const int j = blockIdx.x;
    for (int m = threadIdx.x; m < fast::kPTabIntervals; m += blockDim.x)
        coef[(size_t)j * fast::kPTabIntervals + m] = fast::compute_ptab_coef(curves, j, m + fast::kPTabFirstInterval);
}

constexpr int kPTabThreads = 512;
template <unsigned KINDS, bool QIN>
__global__ void __launch_bounds__(kPTabThreads, 1) suite_fast_ptab_kernel(const __grid_constant__ PColParams prm,
                                                                          const Coef *__restrict__ coef) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t mbar;
    Coef *s_tab = reinterpret_cast<Coef *>(smem_raw);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t row_bytes = fast::kPTabIntervals * sizeof(Coef);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)),
                     "r"(row_bytes * (uint32_t)fast::kPTabNodes) : "memory");
        for (int j = 0; j < fast::kPTabNodes; ++j) {
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                    smem_u32(s_tab + (size_t)j * fast::kPTabIntervals)),
                "l"(coef + (size_t)j * fast::kPTabIntervals), "r"(row_bytes), "r"(smem_u32(&mbar))
                : "memory");
        }
    }
    {
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done) : "r"(smem_u32(&mbar)), "r"(0u) : "memory");
        }
    }
    const fast::PTabView ptab{s_tab, fast::ptab_desc()};
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < prm.n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t col = base + threadIdx.x;
        if (col >= prm.n) continue;
        const PColRd rd{prm.p + col, prm.t + col, prm.td + col, prm.ls, prm.pls};
        fast::FResult res[3];
        fast::NoProfile np;
        fast::NoRing ring;
        const unsigned redo = fast::suite_column_pcol<KINDS, 1, QIN>(rd, prm.L, prm.tb, prm.o, np, ring, ptab, res);
        if (KINDS & 1u) store_fast(prm.outs[0], col, res[0]);
        if (KINDS & 2u) store_fast(prm.outs[1], col, res[1]);
        if (KINDS & 4u) store_fast(prm.outs[2], col, res[2]);
        if (redo) push_redo(prm.list, prm.list_count, prm.n, col, redo);
    }
}

// ---- per-column pressure, v6 sweep (xp_fast_pcol6.cuh): default options, scalar outputs ----------------------
struct PColRd32 {
    const float *p, *t, *td;
    uint32_t col, lstride, plstride;
    __device__ __forceinline__ uint32_t off0() const { return col; }
    __device__ __forceinline__ uint32_t ls() const { return lstride; }
    __device__ __forceinline__ uint32_t pls() const { return plstride; }
    __device__ __forceinline__ float ldP(uint32_t off) const { return XP_LDSTREAM(p + off); }
    __device__ __forceinline__ float ldT(uint32_t off) const { return XP_LDSTREAM(t + off); }
    __device__ __forceinline__ float ldTd(uint32_t off) const { return XP_LDSTREAM(td + off); }
    __device__ __forceinline__ void prefetch(uint32_t offp, uint32_t off) const {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p + offp));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(t + off));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(td + off));
    }
};

// p/T/Td of the lowest levels of every thread's column: element (level k, which, thread) at
// base[(3 k + which) * blockDim.x + thread] -- conflict-free.
struct StashSmem3 {
    float *base;
    int stride, cap;
    __device__ __forceinline__ int capacity() const { return cap; }
    __device__ __forceinline__ void put(int k, float p, float t, float td) {
        base[(3 * k) * stride] = p; base[(3 * k + 1) * stride] = t; base[(3 * k + 2) * stride] = td;
    }
    __device__ __forceinline__ void get(int k, float &p, float &t, float &td) const {
        p = base[(3 * k) * stride]; t = base[(3 * k + 1) * stride]; td = base[(3 * k + 2) * stride];
    }
};

constexpr int kPCol6Threads = 256;
constexpr int kPCol6StashLevels = 8;       // 8 levels x 3 arrays x 4 B x 256 threads = 24 KB per CTA (more levels cost occupancy: measured)

template <unsigned KINDS>
__global__ void __launch_bounds__(kPCol6Threads, 2) suite_fast_pcol6_kernel(const __grid_constant__ PColParams prm,
                                                                            int stash_levels) {
    extern __shared__ __align__(16) float s_stash[];
    const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= prm.n) return;
    const PColRd32 rd{prm.p, prm.t, prm.td, (uint32_t)col, (uint32_t)prm.ls, (uint32_t)prm.pls};
    StashSmem3 st{s_stash + threadIdx.x, (int)blockDim.x, stash_levels};
    fast::FResult res[3];
    const unsigned redo = fast::suite_column_pcol6<KINDS>(rd, prm.L, prm.tb, prm.o, st, res);
    if (KINDS & 1u) store_fast(prm.outs[0], col, res[0]);
    if (KINDS & 2u) store_fast(prm.outs[1], col, res[1]);
    if (KINDS & 4u) store_fast(prm.outs[2], col, res[2]);
    if (redo) push_redo(prm.list, prm.list_count, prm.n, col, redo);
}

}  // namespace

// Build/experiment knobs from the environment, read ONCE per process (thread-safe static initialisation), never
// in the launch path.
struct FastKnobs { int pcol6, staged, sweep, ring, ptab; };
static const FastKnobs &fast_knobs() {
    static const FastKnobs k = [] {
        FastKnobs r;
        const char *e = getenv("XP_PCOL6");
        r.pcol6 = e ? atoi(e) : 0;
        e = getenv("XP_FAST_STAGED");
        r.staged = e ? atoi(e) : 0;          // default 0: measured fastest (DESIGN.md section 6)
        e = getenv("XP_PCOL_RING");
        // 1: re-based profile sweeps read through the shared-memory ring.  Default 0 -- measured on 10 M x 90
        // most-unstable + profile rows: DRAM reads 38.6 -> 24.5 GB, writes 30.5 -> 26.7 GB, but the kernel takes 39.1
        // instead of 33.2 ms (12 instead of 16 warps per SM; it is latency-bound, not DRAM-bound: 2.1 TB/s).
        r.ring = e ? atoi(e) : 0;
        e = getenv("XP_PCOL_TABLE");
        r.ptab = e ? atoi(e) : 1;            // 1: per-column pressure, default options: adiabat family in shared memory
        e = getenv("XP_FAST_SWEEP");
        r.sweep = e ? atoi(e) : 7;           // 7: xp_fast7.cuh (default), 6: xp_fast6.cuh
        return r;
    }();
    return k;
}

size_t fast_scratch_bytes(int64_t n) {
    // Prep | coef table | list counter | list
    return ((sizeof(Prep) + 255) & ~(size_t)255) + (size_t)fast::kMaxLevels * fast::kNI * sizeof(Coef) + 256 +
           3 * (size_t)n * sizeof(uint32_t);
}

static bool wants_profile(int kind_mask, const OutArg<float> *outs) {
    for (int q = 0; q < 3; ++q) {
        if (!((kind_mask >> q) & 1)) continue;
        const OutArg<float> &o = outs[q];
        if (o.prof_p || o.prof_t || o.prof_tv || o.prof_et || o.prof_etv || o.prof_etd) return true;
    }
    return false;
}

bool fast_eligible(const ColsArg<float> &cols, int kind_mask, const OutArg<float> *outs, const Opts &o) {
    if (cols.L < 3 || cols.n >= (int64_t)1 << 28) return false;
    // specific humidity in place of the dewpoint: on a shared axis only the v7 sweep (default options) converts on load
    // (and that sweep addresses the arrays with 32-bit element offsets)
    if (cols.qmode && cols.p1d && (!(o.vtc && o.compat == 141 && o.pos_neg) ||
                                   (uint64_t)cols.n + (uint64_t)cols.L * (uint64_t)cols.ls >= ((uint64_t)1 << 32))) return false;
    if (cols.p1d && cols.L > fast::kMaxLevels) return false;
    if (kind_mask & ~(kSB | kML | kMU)) return false;
    if (cols.p1d && wants_profile(kind_mask, outs)) return false;   // shared-axis kernel: scalars only
    return true;
}

int launch_suite_fast(const ColsArg<float> &cols, const Tables &tb, const Opts &o, int kind_mask,
                      const OutArg<float> *outs, void *scratch, uint32_t *flags, int sm_count,
                      cudaStream_t stream) {
    if (cols.n <= 0) return 0;
    unsigned char *base = static_cast<unsigned char *>(scratch);
    Prep *prep = reinterpret_cast<Prep *>(base);
    size_t off = (sizeof(Prep) + 255) & ~(size_t)255;
    Coef *coef = reinterpret_cast<Coef *>(base + off);
    off += (size_t)fast::kMaxLevels * fast::kNI * sizeof(Coef);
    uint32_t *count = reinterpret_cast<uint32_t *>(base + off);
    off += 256;
    uint32_t *list = reinterpret_cast<uint32_t *>(base + off);

    cudaMemsetAsync(count, 0, 4 * sizeof(uint32_t), stream);
    const int mode = (o.vtc && o.compat == 141 && o.pos_neg) ? 1 : 0;
    ListParams lp;
    lp.cols = cols; lp.tb = tb; lp.o = o;
    lp.o.qmode = cols.qmode;
    for (int q = 0; q < 3; ++q) lp.outs[q] = outs[q];
    lp.list = list; lp.list_count = count; lp.capacity = cols.n; lp.flags = flags;
    if (!cols.p1d) {
        // per-column pressure: no shared-memory table, adiabats gathered from the curve table
        PColParams pp;
        pp.p = cols.p; pp.t = cols.t; pp.td = cols.td; pp.n = cols.n; pp.ls = cols.ls; pp.pls = cols.pls;
        pp.L = cols.L; pp.tb = tb; pp.o = o;
        pp.o.qmode = cols.qmode;
        for (int q = 0; q < 3; ++q) pp.outs[q] = outs[q];
        pp.list = list; pp.list_count = count;
        const unsigned g = (unsigned)((cols.n + kPColThreads - 1) / kPColThreads);
        const bool profile = wants_profile(kind_mask, outs);
        // The v6 sweep for per-column pressure (xp_fast_pcol6.cuh) is kept for experiments (XP_PCOL6=1: surface-based
        // parcel only, 2: every kind).  Measured on the B200 (1 M x 70 SB / 2.8 M x 70 SB+ML, M columns/s): generic
        // sweep 1069 / 693, v6 sweep 938 / 506 -- since the generic sweep reads its pre-pass levels ahead and
        // searches the LCL level in chunks of independent loads it wins everywhere, so it is the default.
        const int pcol6 = fast_knobs().pcol6;
        const uint64_t span = (uint64_t)cols.n + (uint64_t)cols.L * (uint64_t)std::max(cols.ls, cols.pls);
        if (pcol6 && !cols.qmode && ((kind_mask & 7) == 1 || pcol6 == 2) && mode && !profile && span < ((uint64_t)1 << 32)) {
            const int lv = kPCol6StashLevels;
            const size_t smem6 = (size_t)lv * 3 * sizeof(float) * kPCol6Threads;
            const unsigned g6 = (unsigned)((cols.n + kPCol6Threads - 1) / kPCol6Threads);
            // (the shared-memory opt-in is a per-DEVICE attribute: set on every launch, ~1 us, never cached per process)
#define XP_PCOL6_CASE(K)                                                                                          \
    case K:                                                                                                       \
        if (cudaFuncSetAttribute(suite_fast_pcol6_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                 (int)((size_t)kPCol6StashLevels * 3 * sizeof(float) * kPCol6Threads)) != cudaSuccess) return -1; \
        suite_fast_pcol6_kernel<K><<<g6, kPCol6Threads, smem6, stream>>>(pp, lv);                                 \
        break;
            switch (kind_mask & 7) {
                XP_PCOL6_CASE(1) XP_PCOL6_CASE(2) XP_PCOL6_CASE(3) XP_PCOL6_CASE(4) XP_PCOL6_CASE(5) XP_PCOL6_CASE(6) XP_PCOL6_CASE(7)
                default: return -1;
            }
#undef XP_PCOL6_CASE
            launch_suite_list(lp, sm_count, stream);
            return 2;
        }
        // default options, scalar outputs: the adiabat family from shared memory (suite_fast_ptab_kernel)
        // (two or three kinds: +5 % over the gather kernels on 2 M x 70; ONE kind is faster through the gather kernel at
        //  three CTAs per SM -- 1.12 vs 1.02 G columns/s surface-based -- unless XP_PCOL_TABLE=2 forces the table)
        const int nk = ((kind_mask >> 0) & 1) + ((kind_mask >> 1) & 1) + ((kind_mask >> 2) & 1);
        if (mode && !profile && (fast_knobs().ptab == 2 || (fast_knobs().ptab == 1 && nk >= 2))) {
            ptab_coef_kernel<<<fast::kPTabNodes, 160, 0, stream>>>(tb.curves, coef);
            const size_t tsm = (size_t)fast::kPTabNodes * fast::kPTabIntervals * sizeof(Coef);
            const int64_t tiles = (cols.n + kPTabThreads - 1) / kPTabThreads;
            const int gt = (int)(tiles < sm_count ? tiles : sm_count);
#define XP_PTAB_CASE(K)                                                                                               \
    case K:                                                                                                           \
        if (cols.qmode) {                                                                                             \
            if (cudaFuncSetAttribute(suite_fast_ptab_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                                     (int)tsm) != cudaSuccess) return -1;                                             \
            suite_fast_ptab_kernel<K, true><<<gt, kPTabThreads, tsm, stream>>>(pp, coef);                             \
        } else {                                                                                                      \
            if (cudaFuncSetAttribute(suite_fast_ptab_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                     (int)tsm) != cudaSuccess) return -1;                                             \
            suite_fast_ptab_kernel<K, false><<<gt, kPTabThreads, tsm, stream>>>(pp, coef);                            \
        }                                                                                                             \
        break;
            switch (kind_mask & 7) {
                XP_PTAB_CASE(1) XP_PTAB_CASE(2) XP_PTAB_CASE(3) XP_PTAB_CASE(4) XP_PTAB_CASE(5) XP_PTAB_CASE(6) XP_PTAB_CASE(7)
                default: return -1;
            }
#undef XP_PTAB_CASE
            launch_suite_list(lp, sm_count, stream);
            return 3;
        }
        // one LIFTED kind (mixed layer / most unstable) with profile rows: the re-based sweep through the ring
        if (profile && ((kind_mask & 7) == 2 || (kind_mask & 7) == 4) && fast_knobs().ring) {
            const size_t rsm = (size_t)kPColRingLevels * 3 * sizeof(float) * kPColRingThreads;
            const unsigned gr = (unsigned)((cols.n + kPColRingThreads - 1) / kPColRingThreads);
#define XP_PCOL_RING(K, M, Q)                                                                                          \
    do {                                                                                                               \
        if (cudaFuncSetAttribute(suite_fast_pcol_kernel<K, M, true, Q, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                 (int)rsm) != cudaSuccess) return -1;                                                  \
        suite_fast_pcol_kernel<K, M, true, Q, true><<<gr, kPColRingThreads, rsm, stream>>>(pp);                        \
    } while (0)
            if ((kind_mask & 7) == 2) {
                if (cols.qmode) XP_PCOL_RING(2, 0, true); else if (mode) XP_PCOL_RING(2, 1, false); else XP_PCOL_RING(2, 0, false);
            } else {
                if (cols.qmode) XP_PCOL_RING(4, 0, true); else if (mode) XP_PCOL_RING(4, 1, false); else XP_PCOL_RING(4, 0, false);
            }
#undef XP_PCOL_RING
            launch_suite_list(lp, sm_count, stream);
            return 2;
        }
#define XP_PCOL_CASE(K)                                                                          \
    case K:                                                                                      \
        if (cols.qmode) {   /* specific-humidity input: the run-time-option kernels */           \
            if (profile) suite_fast_pcol_kernel<K, 0, true, true><<<g, kPColThreads, 0, stream>>>(pp);   \
            else suite_fast_pcol_kernel<K, 0, false, true><<<g, kPColThreads, 0, stream>>>(pp);  \
        } else if (profile) {                                                                           \
            if (mode) suite_fast_pcol_kernel<K, 1, true><<<g, kPColThreads, 0, stream>>>(pp);    \
            else suite_fast_pcol_kernel<K, 0, true><<<g, kPColThreads, 0, stream>>>(pp);         \
        } else {                                                                                 \
            if (mode) suite_fast_pcol_kernel<K, 1, false><<<g, kPColThreads, 0, stream>>>(pp);   \
            else suite_fast_pcol_kernel<K, 0, false><<<g, kPColThreads, 0, stream>>>(pp);        \
        }                                                                                        \
        break;
        switch (kind_mask & 7) {
            XP_PCOL_CASE(1) XP_PCOL_CASE(2) XP_PCOL_CASE(3) XP_PCOL_CASE(4) XP_PCOL_CASE(5) XP_PCOL_CASE(6) XP_PCOL_CASE(7)
            default: return -1;
        }
#undef XP_PCOL_CASE
        launch_suite_list(lp, sm_count, stream);
        return 2;
    }
    fast_prep_kernel<<<1, 64, 0, stream>>>(cols.p, cols.pls, cols.L, o, prep);

    FastParams fp;
    fp.t = cols.t; fp.td = cols.td; fp.n = cols.n; fp.ls = cols.ls;
    fp.prep = prep; fp.coef = coef; fp.tb = tb; fp.o = o; fp.kinds = (unsigned)kind_mask;
    fp.o.qmode = cols.qmode;
    for (int q = 0; q < 3; ++q) fp.outs[q] = outs[q];
    fp.list = list; fp.list_count = count;
    fp.dense_out = 1;
    for (int q = 0; q < 3; ++q) {
        if (!((kind_mask >> q) & 1)) continue;
        const OutArg<float> &oq = outs[q];
        const bool nine = oq.cape && oq.cin && oq.lcl_p && oq.lcl_t && oq.lcl_tv && oq.lfc_p && oq.lfc_t && oq.el_p && oq.el_t;
        const bool par = oq.par_p && oq.par_t && oq.par_td, no_par = !oq.par_p && !oq.par_t && !oq.par_td;
        if (!nine || oq.shift || (q == 0 ? !no_par : !par)) fp.dense_out = 0;
    }
    // shared memory: Prep | coefficient table | (staged) the environment curve of every thread
    const size_t smem_table = ((sizeof(Prep) + 127) & ~(size_t)127) + (size_t)cols.L * fast::kNI * sizeof(Coef);
    const size_t smem_env = (size_t)cols.L * kFastThreads * sizeof(float);
    int staged = cols.qmode ? 0 : fast_knobs().staged;      // specific-humidity input: the v7 sweep only
    if (staged == 1 && smem_table + smem_env + 256 > (size_t)227 * 1024) staged = 0;
    // the v6 sweep addresses T/Td with 32-bit element offsets; larger arrays take the generic sweep (variant 2)
    if (mode == 1 && staged == 0 && (uint64_t)cols.n + (uint64_t)cols.L * (uint64_t)cols.ls >= ((uint64_t)1 << 32)) staged = 2;
    const bool v6 = (mode == 1 && staged == 0);
    if (v6 && (fast_knobs().sweep == 7 || cols.qmode)) staged = cols.qmode ? 4 : 3;
    if (cols.qmode && staged != 4) return -1;               // (fast_eligible keeps such calls away)
    fast_coef_kernel<<<cols.L, fast::kNI, 0, stream>>>(prep, tb.curves, coef, v6 ? 1 : 0);
    size_t smem = smem_table + (staged == 1 ? smem_env : 0);
    fp.stash_levels = 0;
    if (v6) {
        // v6 / v7 sweep: stash as many of the lowest levels as fit (at most 16: the pre-pass depth of real axes)
        const size_t per_level = 2 * sizeof(float) * kFastThreads;
        const size_t room = (size_t)227 * 1024 - 256 - smem_table;
        int lv = (int)(room / per_level);
        lv = lv > 16 ? 16 : lv;
        fp.stash_levels = lv;
        smem += (size_t)lv * per_level;
    }
    const int threads = kFastThreads;      // one persistent CTA per SM (640 threads x 96 registers: measured best of 512..768)
    const int64_t tiles = (cols.n + threads - 1) / threads;
    const int grid = (int)(tiles < sm_count ? tiles : sm_count);
    // the dynamic shared-memory opt-in is a per-DEVICE function attribute: set it on every launch (a process may
    // hold contexts on several GPUs; a process-wide cache would skip the second device)
#define XP_FAST_LAUNCH(K, M, S)                                                                                  \
    do {                                                                                                         \
        if (cudaFuncSetAttribute(suite_fast_kernel<K, M, kFastThreads, S>,                                       \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)         \
            return -1;                                                                                           \
        suite_fast_kernel<K, M, kFastThreads, S><<<grid, kFastThreads, smem, stream>>>(fp);                      \
    } while (0)
#define XP_FAST_CASE(K)                                                                           \
    case K:                                                                                       \
        if (staged == 1) { if (mode) XP_FAST_LAUNCH(K, 1, 1); else XP_FAST_LAUNCH(K, 0, 1); }     \
        else if (staged == 2) { if (mode) XP_FAST_LAUNCH(K, 1, 2); else XP_FAST_LAUNCH(K, 0, 2); }\
        else if (staged == 3) { XP_FAST_LAUNCH(K, 1, 3); }                                        \
        else if (staged == 4) { XP_FAST_LAUNCH(K, 1, 4); }                                        \
        else { if (mode) XP_FAST_LAUNCH(K, 1, 0); else XP_FAST_LAUNCH(K, 0, 0); }                 \
        break;
    switch (kind_mask & 7) {
        XP_FAST_CASE(1) XP_FAST_CASE(2) XP_FAST_CASE(3) XP_FAST_CASE(4) XP_FAST_CASE(5) XP_FAST_CASE(6) XP_FAST_CASE(7)
        default: return -1;
    }
#undef XP_FAST_LAUNCH
#undef XP_FAST_CASE

    launch_suite_list(lp, sm_count, stream);
    return 4;
}

// ---- float64 columns ---------------------------------------------------------------------------------------------
// The reference computes in float64 (MetPy / pint); callers that hand float64 arrays over get the same v7 kernel: the
// sweep consumes every level rounded to float32 (its decisions keep their margins: the rounding is 1.5e-5 K against
// kDecisionEps = 6e-4 K), the parcels' own T / Td and the mixed-layer sums are read in float64, the outputs are
// written as float64, and the fix-up list is recomputed by the float64 exact code on the float64 columns.
int launch_suite_fast_f64(const ColsArg<double> &cols, const Tables &tb, const Opts &o, int kind_mask,
                          const OutArg<double> *outs, void *scratch, uint32_t *flags, int sm_count,
                          cudaStream_t stream) {
    if (cols.n <= 0) return 0;
    const bool mode1 = o.vtc && o.compat == 141 && o.pos_neg;
    if (!cols.p1d || !mode1 || cols.qmode || cols.L < 3 || cols.L > fast::kMaxLevels || cols.n >= ((int64_t)1 << 28)) return -2;
    if (kind_mask & ~(kSB | kML | kMU)) return -2;
    if ((uint64_t)cols.n + (uint64_t)cols.L * (uint64_t)cols.ls >= ((uint64_t)1 << 32)) return -2;
    for (int q = 0; q < 3; ++q) {
        if (!((kind_mask >> q) & 1)) continue;
        const OutArg<double> &oq = outs[q];
        if (oq.prof_p || oq.prof_t || oq.prof_tv || oq.prof_et || oq.prof_etv || oq.prof_etd) return -2;
    }
    unsigned char *base = static_cast<unsigned char *>(scratch);
    Prep *prep = reinterpret_cast<Prep *>(base);
    size_t off = (sizeof(Prep) + 255) & ~(size_t)255;
    Coef *coef = reinterpret_cast<Coef *>(base + off);
    off += (size_t)fast::kMaxLevels * fast::kNI * sizeof(Coef);
    uint32_t *count = reinterpret_cast<uint32_t *>(base + off);
    off += 256;
    uint32_t *list = reinterpret_cast<uint32_t *>(base + off);
    cudaMemsetAsync(count, 0, 4 * sizeof(uint32_t), stream);
    ListParamsT<double> lp;
    lp.cols = cols; lp.tb = tb; lp.o = o;
    for (int q = 0; q < 3; ++q) lp.outs[q] = outs[q];
    lp.list = list; lp.list_count = count; lp.capacity = cols.n; lp.flags = flags;
    fast_prep_kernel<<<1, 64, 0, stream>>>(cols.p, cols.pls, cols.L, o, prep);
    fast_coef_kernel<<<cols.L, fast::kNI, 0, stream>>>(prep, tb.curves, coef, 1);
    FastParamsT<double> fp;
    fp.t = cols.t; fp.td = cols.td; fp.n = cols.n; fp.ls = cols.ls;
    fp.prep = prep; fp.coef = coef; fp.tb = tb; fp.o = o; fp.kinds = (unsigned)kind_mask;
    fp.o.qmode = 0;
    for (int q = 0; q < 3; ++q) fp.outs[q] = outs[q];
    fp.list = list; fp.list_count = count;
    fp.dense_out = 1;
    for (int q = 0; q < 3; ++q) {
        if (!((kind_mask >> q) & 1)) continue;
        const OutArg<double> &oq = outs[q];
        const bool nine = oq.cape && oq.cin && oq.lcl_p && oq.lcl_t && oq.lcl_tv && oq.lfc_p && oq.lfc_t && oq.el_p && oq.el_t;
        const bool par = oq.par_p && oq.par_t && oq.par_td, no_par = !oq.par_p && !oq.par_t && !oq.par_td;
        if (!nine || oq.shift || (q == 0 ? !no_par : !par)) fp.dense_out = 0;
    }
    const size_t smem_table = ((sizeof(Prep) + 127) & ~(size_t)127) + (size_t)cols.L * fast::kNI * sizeof(Coef);
    const size_t per_level = 2 * sizeof(float) * kFastThreads;
    const size_t room = (size_t)227 * 1024 - 256 - smem_table;
    int lv = (int)(room / per_level);
    lv = lv > 16 ? 16 : lv;
    fp.stash_levels = lv;
    const size_t smem = smem_table + (size_t)lv * per_level;
    const int64_t tiles = (cols.n + kFastThreads - 1) / kFastThreads;
    const int grid = (int)(tiles < sm_count ? tiles : sm_count);
#define XP_FAST64_CASE(K)                                                                                         \
    case K:                                                                                                       \
        if (cudaFuncSetAttribute(suite_fast_kernel<K, 1, kFastThreads, 3, double>,                                \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)          \
            return -1;                                                                                            \
        suite_fast_kernel<K, 1, kFastThreads, 3, double><<<grid, kFastThreads, smem, stream>>>(fp);               \
        break;
    switch (kind_mask & 7) {
        XP_FAST64_CASE(1) XP_FAST64_CASE(2) XP_FAST64_CASE(3) XP_FAST64_CASE(4) XP_FAST64_CASE(5) XP_FAST64_CASE(6) XP_FAST64_CASE(7)
        default: return -1;
    }
#undef XP_FAST64_CASE
    launch_suite_list(lp, sm_count, stream);
    return 4;
}

const uint32_t *fast_list_count_ptr(const void *scratch) {
    const unsigned char *base = static_cast<const unsigned char *>(scratch);
    const size_t off = ((sizeof(Prep) + 255) & ~(size_t)255) + (size_t)fast::kMaxLevels * fast::kNI * sizeof(Coef);
    return reinterpret_cast<const uint32_t *>(base + off) + 3;
}

// number of list entries of the last fast launch (debug/metrics; synchronous copy)
uint32_t fast_last_list_count(void *scratch, cudaStream_t stream) {
    uint32_t v = 0;
    cudaMemcpyAsync(&v, fast_list_count_ptr(scratch), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
    cudaStreamSynchronize(stream);
    return v;
}

}  // namespace xp
