// xp_kernels.cuh -- kernel argument structs and launch prototypes shared by the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "xp_column.cuh"

namespace xp {

// Environment columns in device memory (level-major).
template <typename T>
struct ColsArg {
    const T *p, *t, *td;
    int64_t n;          // columns
    int L;              // levels
    int64_t ls;         // level stride of t/td
    int64_t pls;        // level stride of p
    int p1d;            // pressure is a shared 1-D axis
    int qmode;          // 0: td holds dewpoint; 141 / 162: td holds specific humidity, converted on load in that MetPy form
};

// Outputs of one parcel kind (any pointer may be null).
template <typename T>
struct OutArg {
    T *cape, *cin, *lcl_p, *lcl_t, *lcl_tv, *lfc_p, *lfc_t, *el_p, *el_t;
    T *par_p, *par_t, *par_td;
    int32_t *shift;
    T *prof_p, *prof_t, *prof_tv, *prof_et, *prof_etv, *prof_etd;
    int64_t prof_ls;
    int enabled;
};

template <typename T>
struct ParcelArg {
    const T *p, *t, *td;     // explicit parcel [n]
};

enum KindBits { kSB = 1, kML = 2, kMU = 4, kEX = 8 };

template <typename T>
void launch_cape_cin(const ColsArg<T> &cols, const Tables &tb, const Opts &o, int kind_mask,
                     const OutArg<T> *outs /*[4]: SB, ML, MU, EX*/, const ParcelArg<T> &ex,
                     uint32_t *flags, cudaStream_t stream);

template <typename T>
void launch_lcl(const T *p, const T *t, const T *td, int64_t n, const Opts &o, T *lcl_p, T *lcl_t,
                T *lcl_tv, cudaStream_t stream);

template <typename T>
void launch_moist_lapse(const T *pressure, int64_t ls, int L, int64_t n, const Tables &tb,
                        const T *parcel_t, const T *parcel_p, T *out, int64_t out_ls,
                        cudaStream_t stream);

template <typename T>
void launch_parcel_profile(const T *pressure, int64_t ls, int L, int64_t n, const Tables &tb,
                           const Opts &o, const ParcelArg<T> &parcel, T *out_t, T *out_tv,
                           int64_t out_ls, T *lcl_p, T *lcl_t, T *lcl_tv, cudaStream_t stream);

template <typename T>
void launch_lfc_el(const T *pressure, const T *parcel_t, const T *env_t, int64_t ls, int L,
                   int64_t n, const T *lcl_p, const T *lcl_t, T *lfc_p, T *lfc_t, T *el_p, T *el_t,
                   uint32_t *flags, cudaStream_t stream);

template <typename T>
void launch_cape_cin_base(const T *pressure, const T *env_t, const T *parcel_t, int64_t ls, int L,
                          int64_t n, const T *lfc_p, const T *el_p, const Opts &o, T *cape, T *cin,
                          cudaStream_t stream);

// Exact (float64) recomputation of the (column, parcel kind) items the float32 fast paths hand over.
// `list` has one region of `capacity` entries per kind (SB, ML, MU); an entry is the column index, in
// the SB region OR-ed with kListMuIsSb << 28 when the SB result must also be written to the MU outputs.
// `list_count[0..2]` = entries per kind, `list_count[3]` = columns with at least one entry (device
// memory).  Dense per-kind regions keep every lane of the fix-up kernel busy and its warps kind-uniform.
// Lives in xp_kernels.cu because that file is compiled without FMA contraction.
template <typename T>
struct ListParamsT {
    ColsArg<T> cols;
    Tables tb;
    Opts o;
    OutArg<T> outs[3];
    const uint32_t *list;
    const uint32_t *list_count;
    int64_t capacity;
    uint32_t *flags;
};
using ListParams = ListParamsT<float>;
constexpr unsigned kListMuIsSb = 8u;
constexpr unsigned kListRowsOk = 1u;         // entry >> 28: the float32 profile rows of this item stand (scalars only)

// -DXP_BOUNDS_CHECK (the libxparcel_check.so variant that __graft_entry__.build() also produces; compute-sanitizer is
// closed on the B200 pool): every computed index into the shared-memory stash / coefficient table, the uncertain-column
// list and the T/Td arrays of the fast kernels is checked on the device; a violation prints its site and traps, which
// the host sees as a failed launch (tests/test_gpu_bounds_check.py).
#ifdef XP_BOUNDS_CHECK
#define XP_CHECK(cond)                                                                                     \
    do {                                                                                                   \
        if (!(cond)) {                                                                                     \
            printf("XP_BOUNDS_CHECK failed: %s at %s:%d (block %d thread %d)\n", #cond, __FILE__, __LINE__, \
                   (int)blockIdx.x, (int)threadIdx.x);                                                     \
            __trap();                                                                                      \
        }                                                                                                  \
    } while (0)
#else
#define XP_CHECK(cond) ((void)0)
#endif

// Append the items of one column (redo: bits 0-2 kinds, bit 3 = kListMuIsSb, bits 4-6 = rows-ok per kind).
__device__ __forceinline__ void push_redo(uint32_t *list, uint32_t *count, int64_t capacity, int64_t col,
                                          unsigned redo) {
    XP_CHECK(col >= 0 && col < capacity);
    if (redo & 1u) {
        const uint32_t i = atomicAdd(count + 0, 1u);
        XP_CHECK((int64_t)i < capacity);
        list[i] = (uint32_t)col | ((redo & kListMuIsSb) << 28) | (((redo >> 4) & 1u) << 28);
    }
    if (redo & 2u) {
        const uint32_t i = atomicAdd(count + 1, 1u);
        XP_CHECK((int64_t)i < capacity);
        list[capacity + i] = (uint32_t)col | (((redo >> 5) & 1u) << 28);
    }
    if (redo & 4u) {
        const uint32_t i = atomicAdd(count + 2, 1u);
        XP_CHECK((int64_t)i < capacity);
        list[2 * capacity + i] = (uint32_t)col | (((redo >> 6) & 1u) << 28);
    }
    atomicAdd(count + 3, 1u);
}
// Instrumentation: when set (by run_device around a timed device call, under the context's mutex), launch_suite_list
// records this event on the stream just before the fix-up kernel -- it splits the call's device time into the float32
// sweep (prep + coefficient + sweep kernels) and the float64 fix-up (xp_last_kernel_split_ms).
extern thread_local cudaEvent_t g_event_before_list;
void launch_suite_list(const ListParams &lp, int sm_count, cudaStream_t stream);
void launch_suite_list(const ListParamsT<double> &lp, int sm_count, cudaStream_t stream);   // float64 columns (never staged)

// Float32 fast path of the suite on a shared pressure axis (xp_fast.cu / xp_fast.cuh): prep +
// coefficient + fast kernel + exact fix-up over the uncertain-column list, all on `stream`.
// `scratch` must hold fast_scratch_bytes(n) bytes and must not be shared by launches in flight.
bool fast_eligible(const ColsArg<float> &cols, int kind_mask, const OutArg<float> *outs, const Opts &o);
size_t fast_scratch_bytes(int64_t n);
int launch_suite_fast(const ColsArg<float> &cols, const Tables &tb, const Opts &o, int kind_mask,
                      const OutArg<float> *outs, void *scratch, uint32_t *flags, int sm_count,
                      cudaStream_t stream);
uint32_t fast_last_list_count(void *scratch, cudaStream_t stream);
// device address of that count (columns with at least one list entry) inside `scratch`
const uint32_t *fast_list_count_ptr(const void *scratch);
// The same fast path for float64 columns and outputs on a shared pressure axis with the reference's default options
// (the v7 sweep: float32 per level, float64 parcels; the fix-up list runs on the float64 columns).  Returns the
// number of launches, or -2 when the call does not qualify (the caller then runs the float64 exact kernel).
int launch_suite_fast_f64(const ColsArg<double> &cols, const Tables &tb, const Opts &o, int kind_mask,
                          const OutArg<double> *outs, void *scratch, uint32_t *flags, int sm_count,
                          cudaStream_t stream);

// Derived-index helpers (xp_derived.cu): linear/log interpolation of up to 4 fields at one coordinate
// value per column (PF:1758-1828) and the lowest crossing of a field with a constant (PF:992-1064).
template <typename T>
void launch_interp_levels(const T *coords, int64_t cls, int c1d, const T *const *x, T *const *out, int n_fields,
                          int64_t ls, int L, int64_t n, const T *at, double at_scalar, int log_coords,
                          cudaStream_t stream);
template <typename T>
void launch_level_crossing(const T *x, int64_t xls, int x1d, const T *a, int64_t ls, int L, int64_t n,
                           double level, T *out, cudaStream_t stream);

// Layer primitives (xp_layers.cu): mixed_layer (PF:137-162) of up to 4 variables, mixed_parcel (PF:229-289) with
// all six returned variables (out6 = theta, mixing_ratio, temperature, vapour_pressure, dewpoint, pressure; any
// may be null) and get_layer's bottom/top pressures (PF:63-100, bound_pressure PF:208-227).
template <typename T>
void launch_mixed_layer(const T *p, int64_t pls, int p1d, const T *const *x, T *const *out, int n_fields,
                        int pressure_field, int64_t ls, int L, int64_t n, double depth, cudaStream_t stream);
template <typename T>
void launch_mixed_parcel(const T *p, int64_t pls, int p1d, const T *t, const T *td, int64_t ls, int L, int64_t n,
                         double depth, T *const *out6, cudaStream_t stream);
template <typename T>
void launch_layer_bounds(const T *p, int64_t pls, int p1d, int L, int64_t n, double depth, int interpolate,
                         T *bottom, T *top, cudaStream_t stream);

// Level primitives (xp_levels.cu): insert_level (PF:933-990; outputs [L+1][N]), shift_out_nans (PF:1699-1720),
// trapz (PF:164-206; mask labelled by the lower level, sign +1/-1 = only positive / only negative areas) and the
// pressure-order check of valid_data (PF:2320; ORs kFlagPressure* into `flags`).
template <typename T>
void launch_insert_level(const T *coords, int64_t cls, int c1d, const T *lev_c, const T *const *x,
                         const T *const *lev_x, T *const *out, T *coords_out, int n_fields, int64_t ls, int64_t ols,
                         int L, int64_t n, cudaStream_t stream);
template <typename T>
void launch_shift_out_nans(const T *ref, const T *const *x, T *const *out, int n_fields, int64_t ls, int L,
                           int64_t n, int32_t *shift, cudaStream_t stream);
template <typename T>
void launch_trapz(const T *x, int64_t xls, int x1d, const T *const *v, T *const *out, int n_fields, int64_t ls,
                  int L, int64_t n, const uint8_t *mask, int64_t mls, int sign, cudaStream_t stream);
// find_intersections (PF:992-1064): out6 = all x, all y, increasing x, y, decreasing x, y, each [L-1][N] (row r =
// the interval between levels r and r + 1, the reference's offset label r + 1), any may be null.
template <typename T>
void launch_find_intersections(const T *x, int64_t xls, int x1d, const T *a, const T *b, int64_t ls, int64_t ols,
                               int L, int64_t n, int log_x, T *const *out6, cudaStream_t stream);
// interp1d_numba (PF:23-37) = numpy.interp along the last axis: at/out [rows][m], fp [rows][n], xp [rows][n] or [n].
template <typename T>
void launch_interp1d(const T *at, const T *xp, const T *fp, T *out, int64_t rows, int m, int n, int xp1d,
                     cudaStream_t stream);
// trap_around_zeros (PF:1200-1289): out5 = area, x, dx, x_from, x_to, each [2L-1][N] (rows 0..L-1 = the half-areas
// before a zero, labelled by the lower level; rows L..2L-2 = after it, labelled by the upper level); mask [L][N].
template <typename T>
void launch_trap_around_zeros(const T *x, int64_t xls, int x1d, const T *y, int64_t ls, int64_t ols, int L, int64_t n,
                              int log_x, T *const *out5, uint8_t *mask, cudaStream_t stream);
template <typename T>
void launch_pressure_order(const T *p, int64_t pls, int p1d, int L, int64_t n, uint32_t *flags, cudaStream_t stream);

// Pointwise kernels (xp_derived.cu): q -> Td (PF:1889, 1969), saturation mixing ratio (PF:258, 2047-2053),
// Normand wet-bulb temperature (PF:389-445), significant hail parameter (PF:2261-2306; in6 = mucape, mixing
// ratio, lapse, temp_500, shear, flh) and storm proxies (PF:2323-2407; in13 in the order of ProxyIn in
// xp_derived.cu, 9 uint8 flag arrays in the order of the reference's `proxies` dict, any may be null).
template <typename T>
void launch_dewpoint_from_q(const T *p, const T *t, const T *q, int64_t n, int compat, T *out, cudaStream_t stream);
template <typename T>
void launch_sat_mixing_ratio(const T *p, const T *t, int64_t n, T *out, cudaStream_t stream);
template <typename T>
void launch_dry_lapse(const T *p, const T *t0, const T *p0, int64_t n, T *out, cudaStream_t stream);
template <typename T>
void launch_mixing_ratio(const T *t, const T *td, const T *p, int64_t n, int compat, T *out, cudaStream_t stream);
template <typename T>
void launch_virtual_temperature(const T *t, const T *w, int64_t n, double epsilon, T *out, cudaStream_t stream);
template <typename T>
void launch_wet_bulb(const T *p, const T *t, const T *td, int64_t n, const Tables &tb, T *out, cudaStream_t stream);
template <typename T>
void launch_ship(const T *const *in6, int64_t n, T *out, cudaStream_t stream);
template <typename T>
void launch_storm_proxies(const T *const *in13, uint8_t *const *flags9, T *ship, int64_t n, cudaStream_t stream);

// Downdraft CAPE (xp_downdraft.cu, contract in xp_downdraft.cuh): dcape / start pressure / start temperature [N]
// and the parcel temperature [L][N] with level stride pts; any output may be null.
template <typename T>
void launch_downdraft_cape(const T *p, int64_t pls, int p1d, const T *t, const T *td, int64_t ls, int L, int64_t n,
                           int compat, const Tables &tb, T *dcape, T *p_start, T *t_start, T *parcel_t, int64_t pts,
                           cudaStream_t stream);

// Effective inflow layer (xp_effective.cu, contract in xp_effective.cuh): base / top pressure [N] and, when either
// level output is non-null (all-levels mode), the CAPE / CIN of the parcel of every level [L][N] with level stride
// lls; any output may be null.  `scratch` must hold effective_scratch_bytes(n) bytes and must not be shared by launches
// in flight.  Returns 0, or -1 when a shared pressure axis has too many levels for its ln p table.
size_t effective_scratch_bytes(int64_t n);
template <typename T>
int launch_effective(const ColsArg<T> &cols, const Tables &tb, const Opts &o, double min_cape, double min_cin,
                     T *base, T *top, T *lcape, T *lcin, int64_t lls, uint32_t *flags, void *scratch, int sm_count,
                     cudaStream_t stream);

// Storm kinematics (xp_kinematics.cu, contract in xp_kinematics.cuh): motion6 = Bunkers right u / v, left u / v, mean
// wind u / v; srh4 = SRH over the request's fixed depths; bwd3 = BWD u / v / magnitude; [N] each, any may be null.
// sb / st (SRH layer) and bb / bt (BWD layer) are [N] or null.
struct KinematicsRequest;
template <typename T>
void launch_storm_kinematics(const T *z, const T *u, const T *v, const T *su, const T *sv, int64_t ls, int L,
                             int64_t n, const KinematicsRequest &rq, const T *sb, const T *st, const T *bb,
                             const T *bt, T *const *motion6, T *const *srh4, T *srh_layer, T *const *bwd3,
                             cudaStream_t stream);
// Supercell composite and significant tornado parameters (xp_kinematics.cuh), pointwise over n; scp / stp may be null.
template <typename T>
void launch_composite_parameters(const T *mucape, const T *esrh, const T *ebwd, const T *mlcape, const T *mlcin,
                                 const T *lcl_h, int64_t n, T *scp, T *stp, cudaStream_t stream);

// Table builder (xp_tables.cu): fills index_grid (uint16 [kNP][kNT]) and curves (float
// [kNAdiabats][kNP] ascending pressure).  `scratch_u32` must hold kNP*kNT uint32.
void launch_build_tables(uint16_t *index_grid, float *curves, uint32_t *scratch_u32,
                         cudaStream_t stream);

}  // namespace xp
