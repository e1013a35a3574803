/*
 * xparcel.h -- C ABI of libxparcel.so: B200-native column parcel lifting
 * (LCL -> parcel profile -> LCL insertion -> LFC/EL -> CAPE/CIN for surface-based,
 * mixed-layer and most-unstable parcels).
 *
 * The reference (traupach/xarray_parcel) is pure Python and has no FFI: its boundary for
 * this path is the function surface of modules/parcel_functions.py ("PF").  Each entry
 * point below names the PF function(s) it replaces (file:line); the Python binding a
 * maintainer would add is shown in INTEGRATION.md and implemented in
 * xarray_parcel_b200/_lib.py.
 *
 * Conventions
 *  - Plain pointers and sizes only.  The caller owns every buffer.  No exceptions cross
 *    the ABI: every function returns an xp_status; xp_last_error() gives the message.
 *  - Column data are LEVEL-MAJOR: element (level k, column i) of an array is at
 *    base[k * level_stride + i]; consecutive columns are contiguous so every level read
 *    by a warp is one coalesced line.  Level 0 is the surface; pressure decreases with k.
 *    A (time, level, y, x) C-ordered model field is already level-major per time step.
 *  - Units: hPa and K (PF docstrings, README.md:9).  NaN marks missing data.
 *  - dtype: inputs are float32 or float64; outputs have the dtype of the inputs.
 *    Decision-critical arithmetic is float64 inside the kernels either way.
 *  - mem = XP_MEM_DEVICE: pointers are device pointers on the context's device and the
 *    call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default).
 *    mem = XP_MEM_HOST: pointers are host pointers; the library streams column blocks
 *    (XP_HOST_BLOCK_MB per block, default 192) through three device slots on three streams
 *    (H2D, kernel, D2H of different blocks overlap) and returns when the outputs are
 *    complete.  Page-locked (pinned, cudaHostAlloc / cudaHostRegister) buffers are copied
 *    asynchronously, straight from / to the caller's memory.  Pageable buffers (what NumPy
 *    arrays are) are staged by the library: XP_HOST_THREADS host threads copy each block
 *    between the caller's arrays and a page-locked mirror of its slot, the DMA runs from /
 *    to the mirror, and the outputs of a block are copied out of the mirror when its slot
 *    is reused or the call drains.  Inputs are staged when any of them is pageable;
 *    outputs when the first requested one of cape, cin, lcl/lfc/el/parcel pressure,
 *    level_shift, profile pressure / temperature is -- otherwise they are copied directly.
 *    Column blocks may be slices of wider arrays (level stride > n_columns).
 *  - Reference `assert`s that depend on data (PF:131 'Vertical pressures are not unique',
 *    PF:1149 'Top temperature is NaN.') are reported through xp_take_flags().
 */
#ifndef XPARCEL_H
#define XPARCEL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XP_VERSION_MAJOR 0
#define XP_VERSION_MINOR 1

typedef struct xp_context xp_context; /* one per (process, device): tables + staging buffers */

typedef enum {
    XP_OK = 0,
    XP_ERR_INVALID_ARGUMENT = 1,
    XP_ERR_CUDA = 2,
    XP_ERR_TABLES_NOT_LOADED = 3, /* PF:56-61 'Call load_moist_adiabat_lookups first.' */
    XP_ERR_NO_DEVICE = 4
} xp_status;

typedef enum { XP_F32 = 0, XP_F64 = 1 } xp_dtype;
typedef enum { XP_MEM_DEVICE = 0, XP_MEM_HOST = 1 } xp_memspace;

/* Which parcel is lifted (PF:1477 / PF:1651 / PF:1557 / PF:1394 with explicit parcel). */
typedef enum {
    XP_PARCEL_SURFACE = 0,
    XP_PARCEL_MIXED_LAYER = 1,
    XP_PARCEL_MOST_UNSTABLE = 2,
    XP_PARCEL_EXPLICIT = 3
} xp_parcel_kind;

/* Data-dependent reference assertions, OR-ed over all columns of all calls since the last
 * xp_take_flags(). */
#define XP_FLAG_TOP_TEMPERATURE_NAN 1u     /* PF:1149 */
#define XP_FLAG_PRESSURES_NOT_UNIQUE 2u    /* PF:131  */
#define XP_FLAG_PRESSURE_NOT_DECREASING 4u /* PF:2320, set by xp_valid_data */
#define XP_FLAG_PRESSURE_ORDER_CHECKED 8u  /* xp_valid_data saw at least one non-NaN pressure difference */

/* Environment columns: pressure/temperature/dewpoint [n_levels][n_columns]. */
typedef struct {
    const void *pressure;
    const void *temperature;
    const void *dewpoint;
    int64_t n_columns;
    int32_t n_levels;
    int32_t dtype;                 /* xp_dtype */
    int64_t level_stride;          /* elements between levels of temperature and dewpoint */
    int64_t pressure_level_stride; /* elements between levels of pressure */
    int32_t pressure_is_1d;        /* 1: pressure is one shared axis [n_levels] (ERA5-style
                                      pressure levels); element k at pressure[k*pressure_level_stride] */
    int32_t mem;                   /* xp_memspace, applies to inputs AND outputs of the call */
    int32_t dewpoint_is_specific_humidity;
                                   /* 1: `dewpoint` holds SPECIFIC HUMIDITY q [kg/kg] instead; every kernel converts it as
                                      each level is loaded, Td = metpy.calc.dewpoint_from_specific_humidity(p, T, q) in the
                                      form of xp_options.metpy_compat (the q -> Td front end of conv_properties,
                                      PF:1889, 1969; parcel_test.py:432-436) -- model output (p, T, q) is consumed
                                      directly and the dewpoint array is never materialised.  Parcel dewpoints
                                      (surface, most-unstable level, mixed-layer mean) are converted in float64. */
    int32_t reserved_;             /* must be 0 */
} xp_columns;

/* Function kwargs of the reference that select behaviour (PF:1394-1397, PF:1291-1293). */
typedef struct {
    int32_t virtual_temperature_correction; /* default 1 (PF:1396) */
    int32_t lcl_interp_log;                 /* 1 = 'log' (default, PF:1396), 0 = 'linear' */
    int32_t pos_cape_neg_cin;               /* default 1 (PF:1293) */
    int32_t post_zero_cin;                  /* default 0 (PF:1293) */
    int32_t metpy_compat;                   /* 141 = MetPy 1.4.1 formulas (default), 162 = 1.6.2 */
    int32_t exact_only;                     /* default 0; 1 = always run the float64 exact kernel (no
                                               float32 fast path; see DESIGN.md "fast path") */
    double mixed_layer_depth;               /* hPa, default 100 (PF:1652) */
    double most_unstable_depth;             /* hPa, default 300 (PF:1558) */
} xp_options;

/* Outputs for one parcel kind.  Every pointer is optional (NULL = not written).
 * Scalars are [n_columns]; profile arrays are [n_levels + 1][n_columns] with
 * profile_level_stride elements between levels, NaN-padded at the top. */
typedef struct {
    void *cape, *cin;                                                /* PF:1291-1392, J/kg */
    void *lcl_pressure, *lcl_temperature, *lcl_virtual_temperature;  /* PF:609-682 */
    void *lfc_pressure, *lfc_temperature, *el_pressure, *el_temperature; /* PF:1066-1198 */
    void *parcel_pressure, *parcel_temperature, *parcel_dewpoint;    /* the lifted parcel
                                         (PF:229-289 mixed_parcel / PF:102-135 most_unstable_parcel) */
    int32_t *level_shift; /* number of input levels removed below the lifted column (PF:1551-1553
                             MU: index of the MU level; PF:1636-1638 ML: levels in the mixed layer);
                             n_levels for a column with no valid parcel */
    void *profile_pressure, *profile_temperature, *profile_virtual_temperature;      /* PF:806-931 */
    void *profile_environment_temperature, *profile_environment_virtual_temperature;
    void *profile_environment_dewpoint;
    int64_t profile_level_stride;
} xp_parcel_out;

/* Explicit parcel for XP_PARCEL_EXPLICIT (PF:1394 cape_cin's parcel_* arguments): [n_columns]. */
typedef struct {
    const void *pressure, *temperature, *dewpoint;
} xp_parcel_in;

/* ---- lifetime ------------------------------------------------------------------------ */
const char *xp_version(void);
xp_status xp_create(int device, xp_context **out_ctx);
void xp_destroy(xp_context *ctx);
const char *xp_last_error(const xp_context *ctx); /* ctx may be NULL: last error of xp_create */
xp_status xp_take_flags(xp_context *ctx, void *stream, uint32_t *out_flags); /* syncs `stream` */
void xp_default_options(xp_options *opts);

/* ---- moist-adiabat lookup tables: PF:39-61, 318-356, 447-523 --------------------------
 * index grid uint16 [XP_TABLE_NP (descending pressure 1100..2.5)][XP_TABLE_NT (173..315.98)],
 * 0 = no adiabat; curves float32 [XP_TABLE_NADIABATS][XP_TABLE_NP] on ASCENDING pressure
 * (PF:54 sortby('pressure')). */
#define XP_TABLE_NP 2196
#define XP_TABLE_NT 7150
#define XP_TABLE_NADIABATS 14300
xp_status xp_tables_build(xp_context *ctx, void *stream);   /* replaces moist_adiabat_lookup PF:447-523 */
xp_status xp_tables_set(xp_context *ctx, const uint16_t *index_grid_host, const float *curves_host);
xp_status xp_tables_get(xp_context *ctx, uint16_t *index_grid_host, float *curves_host);
int xp_tables_loaded(const xp_context *ctx);                 /* lookup_tables_loaded PF:56-61 */

/* ---- the fused hot path ----------------------------------------------------------------
 * xp_cape_cin: one parcel kind.  Replaces surface_based_cape_cin (PF:1477-1514),
 * mixed_layer_cape_cin (PF:1651-1697) incl. mix_layer/mixed_parcel/mixed_layer/get_layer,
 * most_unstable_cape_cin (PF:1557-1602) incl. from_most_unstable_parcel/most_unstable_parcel/
 * bound_pressure/shift_out_nans, and cape_cin (PF:1394-1475) for an explicit parcel; inside:
 * lcl, parcel_profile(_with_lcl), moist_lapse, add_lcl_to_profile/insert_level,
 * linear/log_interp, find_intersections, lfc_el, trap_around_zeros, trapz, cape_cin_base.
 * `explicit_parcel` is used only for XP_PARCEL_EXPLICIT. */
xp_status xp_cape_cin(xp_context *ctx, const xp_columns *cols, int32_t kind,
                      const xp_parcel_in *explicit_parcel, const xp_options *opts,
                      const xp_parcel_out *out, void *stream);

/* xp_suite: surface-based + mixed-layer + most-unstable in ONE pass over the columns
 * (the benchmark metric).  out[0]=SB, out[1]=ML, out[2]=MU; an entry may be NULL. */
xp_status xp_suite(xp_context *ctx, const xp_columns *cols, const xp_options *opts,
                   const xp_parcel_out *out_sb, const xp_parcel_out *out_ml,
                   const xp_parcel_out *out_mu, void *stream);

/* ---- individually exposed steps (device memory only) ------------------------------------ */
/* lcl PF:609-682: [n] parcels -> lcl pressure/temperature/virtual temperature. */
xp_status xp_lcl(xp_context *ctx, const void *parcel_pressure, const void *parcel_temperature,
                 const void *parcel_dewpoint, int64_t n, int32_t dtype, const xp_options *opts,
                 void *lcl_pressure, void *lcl_temperature, void *lcl_virtual_temperature,
                 void *stream);
/* moist_lapse PF:525-607: parcel temperature at pressure[k][i] on the adiabat through
 * (parcel_pressure[i], parcel_temperature[i]). */
xp_status xp_moist_lapse(xp_context *ctx, const void *pressure, int64_t level_stride,
                         int32_t n_levels, int64_t n_columns, int32_t dtype,
                         const void *parcel_temperature, const void *parcel_pressure,
                         void *out_temperature, int64_t out_level_stride, void *stream);
/* parcel_profile PF:712-780 (no LCL level): temperature and virtual temperature of the lifted
 * parcel on the input levels. */
xp_status xp_parcel_profile(xp_context *ctx, const void *pressure, int64_t level_stride,
                            int32_t n_levels, int64_t n_columns, int32_t dtype,
                            const xp_parcel_in *parcel, const xp_options *opts,
                            void *out_temperature, void *out_virtual_temperature,
                            int64_t out_level_stride, void *lcl_pressure, void *lcl_temperature,
                            void *lcl_virtual_temperature, void *stream);
/* lfc_el PF:1066-1198 on caller-supplied parcel/environment temperature arrays [m][n]. */
xp_status xp_lfc_el(xp_context *ctx, const void *pressure, const void *parcel_temperature,
                    const void *temperature, int64_t level_stride, int32_t n_levels,
                    int64_t n_columns, int32_t dtype, const void *lcl_pressure,
                    const void *lcl_temperature, void *lfc_pressure, void *lfc_temperature,
                    void *el_pressure, void *el_temperature, void *stream);
/* cape_cin_base PF:1291-1392 (+ trap_around_zeros PF:1200-1289, trapz PF:164-206). */
xp_status xp_cape_cin_base(xp_context *ctx, const void *pressure, const void *temperature,
                           const void *parcel_temperature, int64_t level_stride,
                           int32_t n_levels, int64_t n_columns, int32_t dtype,
                           const void *lfc_pressure, const void *el_pressure,
                           const xp_options *opts, void *cape, void *cin, void *stream);

/* ---- derived convective indices (device memory only) ----------------------------------------
 * xp_interp_levels: linear_interp / log_interp (PF:1758-1828, extrapolate=False) of n_fields <= 4
 * fields [n_levels][n_columns] at ONE coordinate value per column (`at` [n_columns], or NULL to use
 * `at_scalar`): bracketing levels = min{c >= at} / max{c <= at}, duplicated coordinates averaged, an
 * exact hit returns the level value, no extrapolation (NaN).  `coords` is [n_levels][n_columns] or,
 * with coords_is_1d, one shared axis.  log_coords = 1 interpolates in ln(coords) (log_interp).
 * Backs lifted_index (PF:1722), deep_convective_index (PF:1830), isobar_temperature (PF:2193),
 * lapse_rate (PF:2102) and wind_shear (PF:2216). */
xp_status xp_interp_levels(xp_context *ctx, const void *coords, int64_t coords_level_stride,
                           int32_t coords_is_1d, const void *const *fields, void *const *outputs,
                           int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                           int32_t dtype, const void *at, double at_scalar, int32_t log_coords,
                           void *stream);
/* xp_level_crossing: lowest coordinate at which `field` crosses `level` (find_intersections PF:992-1064
 * with log_x = False, then .min): freezing_level_height / melting_level_height (PF:2137-2191). */
xp_status xp_level_crossing(xp_context *ctx, const void *coords, int64_t coords_level_stride,
                            int32_t coords_is_1d, const void *field, int64_t level_stride,
                            int32_t n_levels, int64_t n_columns, int32_t dtype, double level,
                            void *output, void *stream);

/* ---- layer primitives of the parcel selectors (device memory only) -----------------------------------
 * xp_mixed_layer: mixed_layer (PF:137-162) of n_fields <= 4 variables [n_levels][n_columns]: the mass-weighted
 * mean over the lowest `depth` hPa = trapz(x = 'pressure') (PF:164-206) over get_layer(interpolate=True)
 * (PF:63-100; the layer top, bottom - depth, is interpolated in ln p and inserted, PF:85-90) divided by the
 * pressure depth (PF:158-161).  `pressure_field` is the index of the field that is the pressure variable itself
 * (its value at the inserted level is the top pressure, PF:87), or -1.  NaN areas are skipped like xarray's sum; columns must satisfy valid_data
 * (PF:2308-2321: pressure decreasing with the level index), trailing NaN pressures end a column. */
xp_status xp_mixed_layer(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                         int32_t pressure_is_1d, const void *const *fields, void *const *outputs, int32_t n_fields,
                         int32_t pressure_field, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                         int32_t dtype, double depth, void *stream);
/* xp_mixed_parcel: mixed_parcel (PF:229-289) with every variable of the Dataset the reference returns
 * ([n_columns] each, any pointer may be NULL): theta and mixing_ratio (the layer means of PF:253/258),
 * temperature (PF:268), vapour_pressure (PF:275), dewpoint (PF:280) and pressure (= level-0 pressure, PF:287). */
typedef struct xp_mixed_parcel_out {
    void *theta, *mixing_ratio, *temperature, *vapour_pressure, *dewpoint, *pressure;
} xp_mixed_parcel_out;
xp_status xp_mixed_parcel(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                          int32_t pressure_is_1d, const void *temperature, const void *dewpoint,
                          int64_t level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype, double depth,
                          const xp_mixed_parcel_out *out, void *stream);
/* xp_layer_bounds: the pressures that bound get_layer (PF:63-100): bottom = the column's largest pressure
 * (PF:80); top = bottom - depth when interpolate != 0 (PF:84), else bound_pressure (PF:208-227): the level
 * pressure closest to it, the larger one on a tie.  Either output may be NULL. */
xp_status xp_layer_bounds(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                          int32_t pressure_is_1d, int32_t n_levels, int64_t n_columns, int32_t dtype, double depth,
                          int32_t interpolate, void *bottom_pressure, void *top_pressure, void *stream);

/* ---- level primitives (device memory only; every array [n_levels][n_columns] unless noted) ----------------
 * xp_insert_level: insert_level (PF:933-990) of n_fields <= 4 variables: `level_coord` / `level_values[f]`
 * ([n_columns]) are inserted by coordinate VALUE (coordinates >= the new one stay, smaller ones move up one level,
 * an equal coordinate is kept below the new level; NaN coordinates travel as the fill value -999 and come back as
 * NaN).  Outputs have n_levels + 1 levels with stride `out_level_stride`; `coords_out` (or NULL) receives the
 * coordinate variable itself. */
xp_status xp_insert_level(xp_context *ctx, const void *coords, int64_t coords_level_stride, int32_t coords_is_1d,
                          const void *level_coord, const void *const *fields, const void *const *level_values,
                          void *const *outputs, int32_t n_fields, void *coords_out, int64_t level_stride,
                          int64_t out_level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype, void *stream);
/* xp_shift_out_nans: shift_out_nans (PF:1699-1720): every field of a column moves down by the number of leading NaN
 * levels of `ref_field`, NaN-padded at the top; `level_shift` ([n_columns] int32, or NULL) receives that number.
 * Outputs must not alias the inputs. */
xp_status xp_shift_out_nans(xp_context *ctx, const void *ref_field, const void *const *fields, void *const *outputs,
                            int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                            int32_t dtype, int32_t *level_shift, void *stream);
/* xp_trapz: trapz (PF:164-206): per column sum of |x[k+1] - x[k]| * (v[k] + v[k+1]) / 2 over the intervals whose
 * `mask` byte (labelled by the lower level, [>= n_levels - 1][n_columns], or NULL) is non-zero; sign = +1 / -1 keeps
 * only positive / negative areas (only_positive / only_negative), 0 all; NaN areas are skipped. */
xp_status xp_trapz(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *const *fields,
                   void *const *outputs, int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                   int32_t dtype, const uint8_t *mask, int64_t mask_level_stride, int32_t sign, void *stream);
/* xp_find_intersections: find_intersections (PF:992-1064) of the curves a and b over the coordinate x (ln x with
 * log_x): for every interval between neighbouring levels whose sign(a - b) changes (a NaN sign counts as a change,
 * PF:1022) the crossing point by linear interpolation (PF:1046-1050), split by direction (sign of a - b above the
 * crossing, PF:1030).  Outputs are [n_levels - 1][n_columns] with stride out_level_stride (row r = the interval
 * between levels r and r + 1, the reference's offset label r + 1), NaN where there is no crossing; any may be NULL. */
typedef struct xp_intersections_out {
    void *all_intersect_x, *all_intersect_y, *increasing_x, *increasing_y, *decreasing_x, *decreasing_y;
} xp_intersections_out;
xp_status xp_find_intersections(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *a,
                                const void *b, int64_t level_stride, int64_t out_level_stride, int32_t n_levels,
                                int64_t n_columns, int32_t dtype, int32_t log_x, const xp_intersections_out *out,
                                void *stream);
/* xp_trap_around_zeros: trap_around_zeros (PF:1200-1289, start = 0): for every interval in which y crosses zero
 * (find_intersections against 0 over x, ln x with log_x) the two triangles next to the zero.  area / x / dx / x_from /
 * x_to are [2 n_levels - 1][n_columns] with stride out_level_stride: rows 0 .. n_levels-1 the half-area BEFORE the
 * zero, labelled by the lower level of the interval (the last row is NaN), rows n_levels .. 2 n_levels-2 the half-area
 * AFTER it, labelled by the upper level; NaN where there is no zero.  mask [n_levels][n_columns] (contiguous) is 1
 * where the ordinary trapezoid above a level stays in the integral (PF:1285-1287).  Any output may be NULL. */
typedef struct xp_zero_areas_out {
    void *area, *x, *dx, *x_from, *x_to;
    uint8_t *mask;
} xp_zero_areas_out;
xp_status xp_trap_around_zeros(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *y,
                               int64_t level_stride, int64_t out_level_stride, int32_t n_levels, int64_t n_columns,
                               int32_t dtype, int32_t log_x, const xp_zero_areas_out *out, void *stream);
/* xp_interp1d: interp1d_numba (PF:23-37), the reference's only natively compiled function: numpy.interp along the
 * last (contiguous) axis.  at / out are [n_rows][m], fp is [n_rows][n], xp is [n_rows][n] or, with xp_is_1d, one
 * shared [n]; xp must increase.  Points outside xp take the end values (the caller masks them, PF:598-600). */
xp_status xp_interp1d(xp_context *ctx, const void *at, const void *xp, int32_t xp_is_1d, const void *fp, void *out,
                      int64_t n_rows, int32_t m, int32_t n, int32_t dtype, void *stream);
/* xp_valid_data: the pressure check of valid_data (PF:2320: pressure.diff(vert_dim).max() < 0).  ORs
 * XP_FLAG_PRESSURE_NOT_DECREASING (a difference >= 0 exists) and XP_FLAG_PRESSURE_ORDER_CHECKED (a non-NaN
 * difference exists) into the context flags; read them with xp_take_flags(). */
xp_status xp_valid_data(xp_context *ctx, const void *pressure, int64_t pressure_level_stride, int32_t pressure_is_1d,
                        int32_t n_levels, int64_t n_columns, int32_t dtype, void *stream);

/* ---- pointwise helpers around the hot path (callers and front end, SURVEY.md 8f-1..3) -----------------
 * All arrays hold `n` points of `dtype` in device memory (any shape, flattened); one thread per point. */

/* metpy.calc.dewpoint_from_specific_humidity as the reference calls it in conv_properties /
 * min_conv_properties (PF:1889, 1969).  metpy_compat = 141: via relative humidity (MetPy 1.4.1);
 * 162: via the vapour pressure (MetPy >= 1.6, environment_changes_eval.ipynb:278). */
xp_status xp_dewpoint_from_specific_humidity(xp_context *ctx, const void *pressure, const void *temperature,
                                             const void *specific_humidity, int64_t n, int32_t dtype,
                                             int32_t metpy_compat, void *dewpoint, void *stream);
/* metpy.calc.saturation_mixing_ratio(pressure, temperature) (PF:258; mu_mixing_ratio PF:2047-2053). */
xp_status xp_saturation_mixing_ratio(xp_context *ctx, const void *pressure, const void *temperature, int64_t n,
                                     int32_t dtype, void *mixing_ratio, void *stream);
/* dry_lapse (PF:291-316): parcel_temperature * (pressure / parcel_pressure) ** kappa, all three [n]. */
xp_status xp_dry_lapse(xp_context *ctx, const void *pressure, const void *parcel_temperature,
                       const void *parcel_pressure, int64_t n, int32_t dtype, void *temperature, void *stream);
/* mixing_ratio (PF:684-710): relative humidity from the dewpoint, then the mixing ratio from it
 * (metpy_compat 141 / 162: the two MetPy forms of mixing_ratio_from_relative_humidity). */
xp_status xp_mixing_ratio(xp_context *ctx, const void *temperature, const void *dewpoint, const void *pressure,
                          int64_t n, int32_t dtype, int32_t metpy_compat, void *mixing_ratio, void *stream);
/* virtual_temperature (PF:782-804): temperature * (1 + epsilon * mixing_ratio), epsilon = 0.608 in the reference. */
xp_status xp_virtual_temperature(xp_context *ctx, const void *temperature, const void *mixing_ratio, int64_t n,
                                 int32_t dtype, double epsilon, void *virtual_temperature, void *stream);
/* wet_bulb_temperature (PF:389-445, Normand's rule): lcl (PF:609-682) of every point, then moist_lapse
 * (PF:525-607, lookup tables) from the LCL back to the point's pressure.  Needs the tables. */
xp_status xp_wet_bulb_temperature(xp_context *ctx, const void *pressure, const void *temperature,
                                  const void *dewpoint, int64_t n, int32_t dtype, void *wet_bulb, void *stream);
/* xp_downdraft_cape: downdraft CAPE (MetPy's downdraft_cape recipe) per column, device memory only.
 * Contract (DESIGN.md section 3.12): a level is valid when p, T and Td are non-NaN; the downdraft starts at the point
 * of minimum equivalent potential temperature (Bolton) among the valid levels in 700-500 hPa (np.isclose to a bound
 * counts as inside) and the points at exactly 700 / 500 hPa interpolated in ln p where no level is close to a bound
 * (first minimum, the larger pressure, on a tie); the start temperature is the Normand wet bulb there; the parcel
 * descends on the table adiabat nearest to (start pressure, wet bulb) to every valid level at or below the start;
 * dcape = -Rd * trapezoid(Tv_env - Tv_parcel, ln p) from the surface up, in J/kg, not clipped (negative where the
 * parcel is warmer).  A column that cannot bracket 700 and 500 hPa, a NaN theta-e or a table index of 0 gives NaN in
 * every output.  metpy_compat (141 / 162) selects the environment's mixing ratio form as in xp_mixing_ratio.
 * Outputs: dcape [J/kg], start_pressure [hPa], start_temperature [K] ([n_columns] each) and parcel_temperature
 * ([n_levels][n_columns] with level stride parcel_level_stride: the descending parcel, NaN above the start and on
 * invalid levels); a NULL output is skipped.  Needs the tables (XP_ERR_TABLES_NOT_LOADED). */
typedef struct xp_downdraft_out {
    void *dcape, *start_pressure, *start_temperature, *parcel_temperature;
    int64_t parcel_level_stride;
} xp_downdraft_out;
xp_status xp_downdraft_cape(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                            int32_t pressure_is_1d, const void *temperature, const void *dewpoint,
                            int64_t level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype,
                            int32_t metpy_compat, const xp_downdraft_out *out, void *stream);
/* xp_effective_inflow_layer: the effective inflow layer (Thompson et al. 2007; SHARPpy's effective_inflow_layer) per
 * column, device memory only.  Contract (DESIGN.md section 3.13): a level is valid when p, T and Td are non-NaN; the
 * lift from valid level k is the parcel (p_k, T_k, Td_k) on the levels with p <= p_k -- the most-unstable lift with
 * its level forced to k -- with CAPE / CIN per `opts` (virtual_temperature_correction, lcl_interp_log,
 * pos_cape_neg_cin, post_zero_cin, metpy_compat; float64 arithmetic; exact_only and mixed_layer_depth have no effect);
 * a level passes when cape >= min_cape && cin > min_cin (NaN fails).  Gate: the column's most-unstable parcel (over
 * opts->most_unstable_depth) must pass, else base and top are NaN.  Base: the first valid level from the surface up
 * that passes (none: NaN).  Top: the valid level just below the first valid level above the base that fails (NaN if
 * none fails; a one-level layer has top == base).  Outputs, in the input dtype, any may be NULL: base_pressure and
 * top_pressure [n_columns] in hPa (input pressures, copied exactly); level_cape / level_cin [n_levels][n_columns] with
 * level stride level_out_stride: the CAPE / CIN of the parcel of every valid level, NaN on invalid levels -- asking
 * for either lifts EVERY valid level of EVERY column, whatever the gate; base and top are the same in both modes.
 * The most-unstable selection and the lifts report XP_FLAG_PRESSURES_NOT_UNIQUE and XP_FLAG_TOP_TEMPERATURE_NAN through
 * xp_take_flags.  XP_ERR_INVALID_ARGUMENT for mem = XP_MEM_HOST, dewpoint_is_specific_humidity = 1, n_levels < 1 or a
 * non-zero reserved_; XP_ERR_TABLES_NOT_LOADED without the tables. */
typedef struct xp_effective_out {
    void *base_pressure, *top_pressure, *level_cape, *level_cin;
    int64_t level_out_stride;
} xp_effective_out;
xp_status xp_effective_inflow_layer(xp_context *ctx, const xp_columns *cols, const xp_options *opts, double min_cape,
                                    double min_cin, const xp_effective_out *out, void *stream);
/* significant_hail_parameter (PF:2261-2306): units as the reference's arguments (mixing ratio kg/kg,
 * lapse K/km negative for decreasing temperature, temp_500 K, shear m/s, flh m). */
xp_status xp_significant_hail_parameter(xp_context *ctx, const void *mucape, const void *mixing_ratio,
                                        const void *lapse, const void *temp_500, const void *shear,
                                        const void *flh, int64_t n, int32_t dtype, void *ship, void *stream);
/* storm_proxies (PF:2323-2407) on the variables conv_properties returns. */
typedef struct xp_proxy_inputs {
    const void *mixed_100_cape, *mixed_50_cape, *mu_cape, *shear_magnitude;
    const void *mixed_100_lifted_index, *mixed_100_dci;
    const void *positive_shear;            /* `dtype` values, 0 = false (NaN counts as true, like NumPy) */
    const void *mixed_50_cin, *mixed_100_cin, *lapse_rate_700_500, *mu_mixing_ratio, *temp_500, *freezing_level;
} xp_proxy_inputs;
typedef struct xp_proxy_outputs {          /* uint8 [n] each, 1 = proxy triggered; any may be NULL */
    uint8_t *craven2004, *kunz2007, *trapp2007, *marsh2009, *allen2011, *allen2014, *eccel2012, *mohr2013, *ship_0_1;
    void *ship;                            /* `dtype` [n] */
} xp_proxy_outputs;
xp_status xp_storm_proxies(xp_context *ctx, const xp_proxy_inputs *in, int64_t n, int32_t dtype,
                           const xp_proxy_outputs *out, void *stream);

/* ---- instrumentation -------------------------------------------------------------------- */
/* Number of kernels this library has launched on ctx since creation. */
uint64_t xp_launch_count(const xp_context *ctx);
/* Columns of the most recent xp_cape_cin/xp_suite call that took the float32 fast path and were
 * recomputed by the float64 exact kernel because a decision was within the float32 error margin
 * (-1 if that call did not use the fast path).  Synchronises the call's stream.  After a call with
 * mem = XP_MEM_HOST: the sum over all its column blocks (-1 if no block took the fast path). */
xp_status xp_last_exact_count(xp_context *ctx, int64_t *out_count);
/* Device time (ms) of the most recent xp_cape_cin/xp_suite kernel launch with
 * mem = XP_MEM_DEVICE, measured with CUDA events on the launch stream; syncs the stream. */
xp_status xp_last_kernel_ms(xp_context *ctx, float *out_ms);
/* The same interval split at the launch of the float64 fix-up kernel, for a call that took the float32 fast path:
 * out_sweep_ms = axis preparation + coefficient + sweep kernels, out_fixup_ms = the fix-up over the hand-over list
 * (XP_ERR_INVALID_ARGUMENT if the most recent timed call did not take the fast path). */
xp_status xp_last_kernel_split_ms(xp_context *ctx, float *out_sweep_ms, float *out_fixup_ms);

#ifdef __cplusplus
}
#endif
#endif /* XPARCEL_H */
