// xp_api.cu -- the C ABI of libxparcel.so (see include/xparcel.h).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/xparcel.h"
#include "xp_kernels.cuh"

using namespace xp;

namespace {
std::string g_create_error;
}

struct xp_context {
    int device = 0;
    uint16_t *d_index = nullptr;
    float *d_curves = nullptr;
    bool tables = false;
    uint32_t *d_flags = nullptr;
    std::string err;
    uint64_t launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr;     // ev_mid: just before the fix-up kernel of a fast call
    bool ev_valid = false, ev_split = false;
    // host-staging pipeline (mem = XP_MEM_HOST)
    static constexpr int kSlots = 3;     // 4 and 6 slots measured: no change (the path is PCIe-bound)
    cudaStream_t slot_stream[kSlots] = {nullptr, nullptr, nullptr};
    void *slot_buf[kSlots] = {nullptr, nullptr, nullptr};
    size_t slot_bytes = 0;
    // page-locked mirrors of the slots: bounce buffers for callers whose host arrays are PAGEABLE (what NumPy /
    // xarray users hold).  Allocated on the first such call.
    void *slot_pin[kSlots] = {nullptr, nullptr, nullptr};
    size_t slot_pin_bytes = 0;
    int host_threads = 8;
    // fast-path scratch (prep, coefficient table, uncertain-column list), one per stream in use
    struct Scratch { void *ptr = nullptr; size_t bytes = 0; };
    std::map<cudaStream_t, Scratch> scratch;
    cudaStream_t last_fast_stream = nullptr;
    bool last_was_fast = false;
    // XP_MEM_HOST calls: the fix-up list count of every block, copied on the block's slot stream into a page-locked
    // array (one entry per block, read once the call has drained), and the call's total (-1: no block was fast)
    uint32_t *block_count_pin = nullptr;
    size_t block_count_cap = 0;
    bool last_was_host = false;
    int64_t last_host_exact = -1;
    int sm_count = 148;
    // experiment knobs, read from the environment once in xp_create (never in the launch path)
    int vote_mask = 3;
    int host_block_mb = 192;     // column blocks of XP_MEM_HOST calls: 96-192 MB 166 M columns/s on the ERA5 suite, 256 MB 161 M, 64 MB 151 M
    std::mutex mu;
};

// at most this many per-stream scratch buffers are kept; beyond it the others are synchronised and freed
constexpr size_t kMaxScratchStreams = 8;

namespace {

struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
            cudaSetDevice(dev);
            changed = true;
        }
    }
    ~DeviceGuard() {
        if (changed) cudaSetDevice(prev);
    }
};

xp_status fail(xp_context *ctx, xp_status st, const std::string &msg) {
    if (ctx) ctx->err = msg;
    else g_create_error = msg;
    return st;
}

xp_status check_cuda(xp_context *ctx, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return XP_OK;
    return fail(ctx, XP_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define XP_CUDA(ctx, call)                                            \
    do {                                                              \
        xp_status _st = check_cuda((ctx), (call), #call);             \
        if (_st != XP_OK) return _st;                                 \
    } while (0)

Opts to_opts(const xp_context *ctx, const xp_options *o) {
    xp_options d;
    xp_default_options(&d);
    if (o) d = *o;
    Opts r;
    r.vtc = d.virtual_temperature_correction != 0;
    r.log_interp = d.lcl_interp_log != 0;
    r.pos_neg = d.pos_cape_neg_cin != 0;
    r.post_zero = d.post_zero_cin != 0;
    r.compat = d.metpy_compat == 162 ? 162 : 141;
    r.ml_depth = d.mixed_layer_depth;
    r.mu_depth = d.most_unstable_depth;
    r.exact_only = d.exact_only != 0;
    r.vote_mask = ctx ? ctx->vote_mask : 3;
    return r;
}

template <typename T>
OutArg<T> to_out(const xp_parcel_out *o) {
    OutArg<T> r;
    std::memset(&r, 0, sizeof(r));
    if (!o) return r;
    r.enabled = 1;
    r.cape = (T *)o->cape; r.cin = (T *)o->cin;
    r.lcl_p = (T *)o->lcl_pressure; r.lcl_t = (T *)o->lcl_temperature;
    r.lcl_tv = (T *)o->lcl_virtual_temperature;
    r.lfc_p = (T *)o->lfc_pressure; r.lfc_t = (T *)o->lfc_temperature;
    r.el_p = (T *)o->el_pressure; r.el_t = (T *)o->el_temperature;
    r.par_p = (T *)o->parcel_pressure; r.par_t = (T *)o->parcel_temperature;
    r.par_td = (T *)o->parcel_dewpoint;
    r.shift = o->level_shift;
    r.prof_p = (T *)o->profile_pressure; r.prof_t = (T *)o->profile_temperature;
    r.prof_tv = (T *)o->profile_virtual_temperature;
    r.prof_et = (T *)o->profile_environment_temperature;
    r.prof_etv = (T *)o->profile_environment_virtual_temperature;
    r.prof_etd = (T *)o->profile_environment_dewpoint;
    r.prof_ls = o->profile_level_stride;
    return r;
}

template <typename T>
ColsArg<T> to_cols(const xp_columns *c, const Opts &o) {
    ColsArg<T> r;
    r.qmode = c->dewpoint_is_specific_humidity ? o.compat : 0;
    r.p = (const T *)c->pressure; r.t = (const T *)c->temperature; r.td = (const T *)c->dewpoint;
    r.n = c->n_columns; r.L = c->n_levels;
    r.ls = c->level_stride; r.pls = c->pressure_level_stride; r.p1d = c->pressure_is_1d != 0;
    return r;
}

xp_status validate_cols(xp_context *ctx, const xp_columns *c) {
    if (!c) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "columns is NULL");
    if (c->n_columns == 0 && c->n_levels >= 1) return XP_OK;      // empty input: nothing to do (pointers may be NULL)
    if (!c->pressure || !c->temperature || !c->dewpoint)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "pressure/temperature/dewpoint must not be NULL");
    if (c->n_levels < 1 || c->n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "n_levels must be >= 1 and n_columns >= 0");
    if (c->dtype != XP_F32 && c->dtype != XP_F64)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "dtype must be XP_F32 or XP_F64");
    if (c->level_stride < c->n_columns)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "level_stride must be >= n_columns");
    if (!c->pressure_is_1d && c->pressure_level_stride < c->n_columns)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "pressure_level_stride must be >= n_columns");
    if (c->mem != XP_MEM_DEVICE && c->mem != XP_MEM_HOST)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "mem must be XP_MEM_DEVICE or XP_MEM_HOST");
    return XP_OK;
}

// The context's scratch buffer of `stream`, grown to at least `need` bytes.  One buffer per stream in use: a call
// may reuse it as soon as the previous call on the same stream is done with it, which stream order guarantees.
cudaError_t stream_scratch(xp_context *ctx, cudaStream_t stream, size_t need, void **out) {
    if (!ctx->scratch.count(stream) && ctx->scratch.size() >= kMaxScratchStreams) {
        // bound the per-stream scratch map: drop the buffers of the other streams (after their work is done)
        for (auto &kv : ctx->scratch) {
            if (kv.second.ptr) { cudaStreamSynchronize(kv.first); cudaFree(kv.second.ptr); }
        }
        ctx->scratch.clear();
    }
    xp_context::Scratch &sc = ctx->scratch[stream];
    if (sc.bytes < need) {
        if (sc.ptr) { cudaStreamSynchronize(stream); cudaFree(sc.ptr); sc.ptr = nullptr; sc.bytes = 0; }
        const cudaError_t e = cudaMalloc(&sc.ptr, need);
        if (e != cudaSuccess) return e;
        sc.bytes = need;
    }
    *out = sc.ptr;
    return cudaSuccess;
}

// Launch the fused kernel on device-resident columns.
template <typename T>
xp_status run_device(xp_context *ctx, const xp_columns *cols, int kind_mask,
                     const xp_parcel_out *const outs[4], const xp_parcel_in *ex, const Opts &o,
                     cudaStream_t stream, bool time_it) {
    OutArg<T> oa[4];
    for (int i = 0; i < 4; ++i) oa[i] = to_out<T>(((kind_mask >> i) & 1) ? outs[i] : nullptr);
    ParcelArg<T> pa = {nullptr, nullptr, nullptr};
    if (kind_mask & kEX) {
        if (!ex || !ex->pressure || !ex->temperature || !ex->dewpoint)
            return fail(ctx, XP_ERR_INVALID_ARGUMENT, "explicit parcel arrays are required");
        pa.p = (const T *)ex->pressure; pa.t = (const T *)ex->temperature; pa.td = (const T *)ex->dewpoint;
    }
    Tables tb = {ctx->d_index, ctx->d_curves};
    ctx->last_was_fast = false;
    if constexpr (std::is_same<T, float>::value) {
        const ColsArg<float> ca = to_cols<float>(cols, o);
        if (!o.exact_only && cols->n_columns > 0 && fast_eligible(ca, kind_mask, oa, o)) {
            void *sp = nullptr;
            XP_CUDA(ctx, stream_scratch(ctx, stream, fast_scratch_bytes(cols->n_columns), &sp));
            if (time_it) { cudaEventRecord(ctx->ev0, stream); g_event_before_list = ctx->ev_mid; }
            const int nl = launch_suite_fast(ca, tb, o, kind_mask, oa, sp, ctx->d_flags, ctx->sm_count, stream);
            g_event_before_list = nullptr;
            if (nl < 0) return check_cuda(ctx, cudaGetLastError(), "fast suite shared-memory attribute");
            ctx->launches += nl;
            if (time_it) { cudaEventRecord(ctx->ev1, stream); ctx->ev_valid = true; ctx->ev_split = nl > 0; }
            ctx->last_was_fast = true;
            ctx->last_fast_stream = stream;
            return check_cuda(ctx, cudaGetLastError(), "fast suite launch");
        }
    }
    if constexpr (std::is_same<T, double>::value) {
        // float64 columns on a shared pressure axis, default options: the same fast kernel (launch_suite_fast_f64)
        if (!o.exact_only && cols->n_columns > 0 && cols->pressure_is_1d && !(kind_mask & kEX)) {
            void *sp = nullptr;
            XP_CUDA(ctx, stream_scratch(ctx, stream, fast_scratch_bytes(cols->n_columns), &sp));
            if (time_it) { cudaEventRecord(ctx->ev0, stream); g_event_before_list = ctx->ev_mid; }
            const int nl = launch_suite_fast_f64(to_cols<double>(cols, o), tb, o, kind_mask, oa, sp, ctx->d_flags,
                                                 ctx->sm_count, stream);
            g_event_before_list = nullptr;
            if (nl == -1) return check_cuda(ctx, cudaGetLastError(), "fast suite shared-memory attribute");
            if (nl >= 0) {
                ctx->launches += nl;
                if (time_it) { cudaEventRecord(ctx->ev1, stream); ctx->ev_valid = true; ctx->ev_split = nl > 0; }
                ctx->last_was_fast = true;
                ctx->last_fast_stream = stream;
                return check_cuda(ctx, cudaGetLastError(), "fast suite launch (float64 columns)");
            }
        }
    }
    if (time_it) { cudaEventRecord(ctx->ev0, stream); ctx->ev_split = false; }
    launch_cape_cin<T>(to_cols<T>(cols, o), tb, o, kind_mask, oa, pa, ctx->d_flags, stream);
    if (time_it) { cudaEventRecord(ctx->ev1, stream); ctx->ev_valid = true; }
    ctx->launches += (cols->n_columns > 0) ? 1 : 0;
    return check_cuda(ctx, cudaGetLastError(), "cape_cin kernel launch");
}

size_t elt_size(int dtype) { return dtype == XP_F64 ? 8 : 4; }

// ---- pageable host memory ------------------------------------------------------------------------------------
// A copy engine can only read page-locked memory.  Given a pageable pointer the driver stages the copy through its
// own small bounce buffer, synchronously (measured on the B200 box: 13.7 GB/s instead of 55 GB/s, and no overlap
// with the kernels).  run_host therefore stages such arrays itself: host threads copy each column block between the
// caller's arrays and a page-locked mirror of the device slot (46 GB/s measured), the DMA runs from / to the
// mirror, and the host copy of one block overlaps the transfers and kernels of the others.
bool is_pageable(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

struct RowCopy { char *dst; const char *src; size_t width, dpitch, spitch; int rows; };

// memcpy of row sets on `nthreads` host threads (rows are cut into <= 4 MB pieces dealt round-robin)
void parallel_copy(const std::vector<RowCopy> &jobs, int nthreads) {
    struct Piece { char *d; const char *s; size_t n; };
    std::vector<Piece> pieces;
    const size_t kPiece = (size_t)4 << 20;
    for (const RowCopy &j : jobs)
        for (int r = 0; r < j.rows; ++r)
            for (size_t o = 0; o < j.width; o += kPiece)
                pieces.push_back({j.dst + (size_t)r * j.dpitch + o, j.src + (size_t)r * j.spitch + o,
                                  std::min(kPiece, j.width - o)});
    if (pieces.empty()) return;
    nthreads = std::max(1, std::min<int>(nthreads, (int)pieces.size()));
    auto work = [&](int t) {
        for (size_t i = t; i < pieces.size(); i += nthreads) std::memcpy(pieces[i].d, pieces[i].s, pieces[i].n);
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
}

// Host-resident columns: stream column blocks through the device (H2D, kernel, D2H on
// kSlots streams so copies of one block overlap the kernel of another).
xp_status run_host(xp_context *ctx, const xp_columns *cols, int kind_mask,
                   const xp_parcel_out *const outs[4], const xp_parcel_in *ex, const Opts &o) {
    const size_t es = elt_size(cols->dtype);
    const int L = cols->n_levels;
    const int64_t N = cols->n_columns;
    ctx->last_host_exact = -1;
    if (N == 0) return XP_OK;
    // per-column device bytes: inputs + every requested output
    size_t per_col = (size_t)(cols->pressure_is_1d ? 2 : 3) * L * es;
    int n_scalar[4] = {0, 0, 0, 0}, n_prof[4] = {0, 0, 0, 0};
    for (int k = 0; k < 4; ++k) {
        if (!((kind_mask >> k) & 1) || !outs[k]) continue;
        const xp_parcel_out *q = outs[k];
        void *sc[] = {q->cape, q->cin, q->lcl_pressure, q->lcl_temperature, q->lcl_virtual_temperature,
                      q->lfc_pressure, q->lfc_temperature, q->el_pressure, q->el_temperature,
                      q->parcel_pressure, q->parcel_temperature, q->parcel_dewpoint};
        for (void *p : sc) n_scalar[k] += p ? 1 : 0;
        void *pr[] = {q->profile_pressure, q->profile_temperature, q->profile_virtual_temperature,
                      q->profile_environment_temperature, q->profile_environment_virtual_temperature,
                      q->profile_environment_dewpoint};
        for (void *p : pr) n_prof[k] += p ? 1 : 0;
        per_col += (size_t)n_scalar[k] * es + (q->level_shift ? 4 : 0) + (size_t)n_prof[k] * (L + 1) * es;
    }
    if (kind_mask & kEX) per_col += 3 * es;
    // block size: ~256 MB per slot (XP_HOST_BLOCK_MB overrides), multiple of 1024 columns.  Measured on the B200
    // box (ERA5 suite, 1.33 GB per call): 256 MB 160.6 M columns/s, 128 MB 155.5, 64 MB 151.3, 32 MB 126.3 --
    // the per-block copies (2 strided H2D, ~40 D2H) cost more than the shorter pipeline fill/drain saves.
    const int block_mb = ctx->host_block_mb;
    int64_t C = (int64_t)((size_t)block_mb << 20) / (int64_t)per_col;
    C = std::max<int64_t>(1024, (C / 1024) * 1024);
    C = std::min<int64_t>(C, ((N + 1023) / 1024) * 1024);
    // every carved array is padded to 256 B: at most 3 inputs + 3 explicit + 4 x (12 scalars + shift + 6
    // profiles) = 82 arrays
    const size_t need = (size_t)C * per_col + 96 * 256;
    if (need > ctx->slot_bytes) {
        for (int s = 0; s < xp_context::kSlots; ++s) {
            if (ctx->slot_buf[s]) { cudaFree(ctx->slot_buf[s]); ctx->slot_buf[s] = nullptr; }
        }
        ctx->slot_bytes = 0;
        for (int s = 0; s < xp_context::kSlots; ++s) XP_CUDA(ctx, cudaMalloc(&ctx->slot_buf[s], need));
        ctx->slot_bytes = need;
    }
    for (int s = 0; s < xp_context::kSlots; ++s)
        if (!ctx->slot_stream[s]) XP_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
    // pageable caller arrays are staged through page-locked mirrors of the slots (see is_pageable above)
    bool stage_in = is_pageable(cols->temperature) || is_pageable(cols->dewpoint) || is_pageable(cols->pressure);
    if ((kind_mask & kEX) && ex) stage_in = stage_in || is_pageable(ex->temperature);
    bool stage_out = false;
    for (int k = 0; k < 4; ++k) {
        if (!((kind_mask >> k) & 1) || !outs[k]) continue;
        const xp_parcel_out *q = outs[k];
        const void *any[] = {q->cape, q->cin, q->lcl_pressure, q->lfc_pressure, q->el_pressure, q->parcel_pressure,
                             q->level_shift, q->profile_pressure, q->profile_temperature};
        for (const void *ptr : any)
            if (ptr) { stage_out = stage_out || is_pageable(ptr); break; }
    }
    if ((stage_in || stage_out) && need > ctx->slot_pin_bytes) {
        for (int s = 0; s < xp_context::kSlots; ++s) {
            if (ctx->slot_pin[s]) { cudaFreeHost(ctx->slot_pin[s]); ctx->slot_pin[s] = nullptr; }
        }
        ctx->slot_pin_bytes = 0;
        for (int s = 0; s < xp_context::kSlots; ++s) XP_CUDA(ctx, cudaHostAlloc(&ctx->slot_pin[s], need, cudaHostAllocDefault));
        ctx->slot_pin_bytes = need;
    }
    // 4 bytes per block of >= 1024 columns: at most 1/2048 of the call's input bytes
    const size_t n_blocks = (size_t)((N + C - 1) / C);
    if (n_blocks > ctx->block_count_cap) {
        if (ctx->block_count_pin) { cudaFreeHost(ctx->block_count_pin); ctx->block_count_pin = nullptr; }
        ctx->block_count_cap = 0;
        const size_t cap = std::max<size_t>(64, n_blocks);
        XP_CUDA(ctx, cudaHostAlloc((void **)&ctx->block_count_pin, cap * sizeof(uint32_t), cudaHostAllocDefault));
        ctx->block_count_cap = cap;
    }
    std::vector<char> block_fast(n_blocks, 0);
    // outputs of a block that wait in the page-locked mirror of its slot until the slot's stream has drained
    std::vector<RowCopy> pending_out[xp_context::kSlots];
    auto retire = [&](int s) -> xp_status {
        if (!stage_in && !stage_out) return XP_OK;
        XP_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[s]));       // the mirror is free again / its outputs are in
        if (!pending_out[s].empty()) { parallel_copy(pending_out[s], ctx->host_threads); pending_out[s].clear(); }
        return XP_OK;
    };

    if ((kind_mask & kEX) && (!ex || !ex->pressure || !ex->temperature || !ex->dewpoint))
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "explicit parcel arrays are required");
    // Whatever way this function is left, no copy may still be writing the caller's buffers and no kernel may
    // still be using the slot buffers: drain every slot stream on exit (error paths included).
    struct DrainSlots {
        xp_context *c;
        ~DrainSlots() {
            for (int s = 0; s < xp_context::kSlots; ++s)
                if (c->slot_stream[s]) cudaStreamSynchronize(c->slot_stream[s]);
        }
    } drain{ctx};
    const char *hp = (const char *)cols->pressure, *ht = (const char *)cols->temperature,
               *htd = (const char *)cols->dewpoint;
    int slot = 0;
    int64_t blk = 0;
    for (int64_t c0 = 0; c0 < N; c0 += C, slot = (slot + 1) % xp_context::kSlots, ++blk) {
        const int64_t n = std::min<int64_t>(C, N - c0);
        cudaStream_t st = ctx->slot_stream[slot];
        char *base = (char *)ctx->slot_buf[slot];
        char *pin = (char *)ctx->slot_pin[slot];
        { const xp_status rs = retire(slot); if (rs != XP_OK) return rs; }
        std::vector<RowCopy> in_jobs;
        size_t off = 0;
        auto carve = [&](size_t bytes) { char *p = base + off; off += (bytes + 255) & ~(size_t)255; return p; };
        // the slot's previous block must be fully drained (its D2H copies are on the same stream,
        // so stream order already guarantees it)
        xp_columns dc = *cols;
        dc.mem = XP_MEM_DEVICE;
        dc.n_columns = n;
        dc.level_stride = n;
        char *dT = carve((size_t)L * n * es), *dTd = carve((size_t)L * n * es), *dP;
        // a host array [rows][width] with pitch `spitch` -> the device carve `d` (contiguous rows)
        struct H2D { char *d; const char *h; size_t width, spitch; int rows; };
        std::vector<H2D> h2d;
        h2d.push_back({dT, ht + c0 * es, (size_t)n * es, (size_t)cols->level_stride * es, L});
        h2d.push_back({dTd, htd + c0 * es, (size_t)n * es, (size_t)cols->level_stride * es, L});
        if (cols->pressure_is_1d) {
            dP = carve((size_t)L * es);
            h2d.push_back({dP, hp, es, (size_t)cols->pressure_level_stride * es, L});
            dc.pressure_level_stride = 1;
        } else {
            dP = carve((size_t)L * n * es);
            h2d.push_back({dP, hp + c0 * es, (size_t)n * es, (size_t)cols->pressure_level_stride * es, L});
            dc.pressure_level_stride = n;
        }
        dc.pressure = dP; dc.temperature = dT; dc.dewpoint = dTd;
        xp_parcel_in dex = {nullptr, nullptr, nullptr};
        if (kind_mask & kEX) {
            const void *src[3] = {ex->pressure, ex->temperature, ex->dewpoint};
            const void **dst[3] = {&dex.pressure, &dex.temperature, &dex.dewpoint};
            for (int i = 0; i < 3; ++i) {
                char *d = carve((size_t)n * es);
                h2d.push_back({d, (const char *)src[i] + c0 * es, (size_t)n * es, 0, 1});
                *dst[i] = d;
            }
        }
        if (stage_in) {
            // caller -> page-locked mirror (host threads), then ONE contiguous DMA per array
            for (const H2D &c : h2d) in_jobs.push_back({pin + (c.d - base), c.h, c.width, c.width, c.spitch, c.rows});
            parallel_copy(in_jobs, ctx->host_threads);
            for (const H2D &c : h2d)
                XP_CUDA(ctx, cudaMemcpyAsync(c.d, pin + (c.d - base), c.width * c.rows, cudaMemcpyHostToDevice, st));
        } else {
            for (const H2D &c : h2d) {
                if (c.rows == 1)
                    XP_CUDA(ctx, cudaMemcpyAsync(c.d, c.h, c.width, cudaMemcpyHostToDevice, st));
                else
                    XP_CUDA(ctx, cudaMemcpy2DAsync(c.d, c.width, c.h, c.spitch, c.width, c.rows, cudaMemcpyHostToDevice, st));
            }
        }
        // device-side outputs mirror the host layout per block
        xp_parcel_out dout[4];
        const xp_parcel_out *douts[4] = {nullptr, nullptr, nullptr, nullptr};
        struct Copy { char *d; char *h; size_t width; size_t hpitch; int rows; };
        std::vector<Copy> copies;
        for (int k = 0; k < 4; ++k) {
            if (!((kind_mask >> k) & 1) || !outs[k]) continue;
            const xp_parcel_out *q = outs[k];
            xp_parcel_out &d = dout[k];
            std::memset(&d, 0, sizeof(d));
            void *const hs[] = {q->cape, q->cin, q->lcl_pressure, q->lcl_temperature,
                                q->lcl_virtual_temperature, q->lfc_pressure, q->lfc_temperature,
                                q->el_pressure, q->el_temperature, q->parcel_pressure,
                                q->parcel_temperature, q->parcel_dewpoint};
            void **ds[] = {&d.cape, &d.cin, &d.lcl_pressure, &d.lcl_temperature,
                           &d.lcl_virtual_temperature, &d.lfc_pressure, &d.lfc_temperature,
                           &d.el_pressure, &d.el_temperature, &d.parcel_pressure,
                           &d.parcel_temperature, &d.parcel_dewpoint};
            for (int i = 0; i < 12; ++i) {
                if (!hs[i]) continue;
                char *p = carve((size_t)n * es);
                *ds[i] = p;
                copies.push_back({p, (char *)hs[i] + c0 * es, (size_t)n * es, 0, 1});
            }
            if (q->level_shift) {
                char *p = carve((size_t)n * 4);
                d.level_shift = (int32_t *)p;
                copies.push_back({p, (char *)q->level_shift + c0 * 4, (size_t)n * 4, 0, 1});
            }
            void *const hpv[] = {q->profile_pressure, q->profile_temperature,
                                 q->profile_virtual_temperature, q->profile_environment_temperature,
                                 q->profile_environment_virtual_temperature,
                                 q->profile_environment_dewpoint};
            void **dpv[] = {&d.profile_pressure, &d.profile_temperature,
                            &d.profile_virtual_temperature, &d.profile_environment_temperature,
                            &d.profile_environment_virtual_temperature,
                            &d.profile_environment_dewpoint};
            d.profile_level_stride = n;
            for (int i = 0; i < 6; ++i) {
                if (!hpv[i]) continue;
                char *p = carve((size_t)(L + 1) * n * es);
                *dpv[i] = p;
                copies.push_back({p, (char *)hpv[i] + c0 * es, (size_t)n * es,
                                  (size_t)q->profile_level_stride * es, L + 1});
            }
            douts[k] = &d;
        }
        xp_status stt = (cols->dtype == XP_F32)
                            ? run_device<float>(ctx, &dc, kind_mask, douts, &dex, o, st, false)
                            : run_device<double>(ctx, &dc, kind_mask, douts, &dex, o, st, false);
        if (stt != XP_OK) return stt;
        if (ctx->last_was_fast) {
            // the block's hand-over count, before the next fast block on this stream resets it in the scratch
            XP_CUDA(ctx, cudaMemcpyAsync(ctx->block_count_pin + blk, fast_list_count_ptr(ctx->scratch[st].ptr),
                                         sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            block_fast[blk] = 1;
        }
        for (const Copy &c : copies) {
            if (stage_out) {
                // device -> page-locked mirror now; mirror -> caller when the slot is retired
                XP_CUDA(ctx, cudaMemcpyAsync(pin + (c.d - base), c.d, c.width * c.rows, cudaMemcpyDeviceToHost, st));
                pending_out[slot].push_back({c.h, pin + (c.d - base), c.width, c.rows == 1 ? c.width : c.hpitch, c.width, c.rows});
            } else if (c.rows == 1) {
                XP_CUDA(ctx, cudaMemcpyAsync(c.h, c.d, c.width, cudaMemcpyDeviceToHost, st));
            } else {
                XP_CUDA(ctx, cudaMemcpy2DAsync(c.h, c.hpitch, c.d, c.width, c.width, c.rows,
                                               cudaMemcpyDeviceToHost, st));
            }
        }
    }
    // drain in block order: the slot after the last one used holds the oldest block in flight
    for (int i = 0; i < xp_context::kSlots; ++i) {
        const int s = (slot + i) % xp_context::kSlots;
        XP_CUDA(ctx, cudaStreamSynchronize(ctx->slot_stream[s]));
        if (!pending_out[s].empty()) { parallel_copy(pending_out[s], ctx->host_threads); pending_out[s].clear(); }
    }
    for (size_t b = 0; b < n_blocks; ++b)
        if (block_fast[b]) ctx->last_host_exact = std::max<int64_t>(ctx->last_host_exact, 0) + ctx->block_count_pin[b];
    return XP_OK;
}

xp_status run_any(xp_context *ctx, const xp_columns *cols, int kind_mask,
                  const xp_parcel_out *const outs[4], const xp_parcel_in *ex, const xp_options *opts,
                  void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    xp_status st = validate_cols(ctx, cols);
    if (st != XP_OK) return st;
    if (!ctx->tables)
        return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (cols->n_columns == 0) return XP_OK;
    DeviceGuard guard(ctx->device);
    const Opts o = to_opts(ctx, opts);
    ctx->last_was_host = cols->mem == XP_MEM_HOST;
    if (cols->mem == XP_MEM_HOST) return run_host(ctx, cols, kind_mask, outs, ex, o);
    if (cols->dtype == XP_F32)
        return run_device<float>(ctx, cols, kind_mask, outs, ex, o, (cudaStream_t)stream, true);
    return run_device<double>(ctx, cols, kind_mask, outs, ex, o, (cudaStream_t)stream, true);
}

}  // namespace

// ================================================================================ C ABI
extern "C" {

const char *xp_version(void) { return "xparcel-b200 0.1 (sm_100a)"; }

void xp_default_options(xp_options *o) {
    if (!o) return;
    o->virtual_temperature_correction = 1;
    o->lcl_interp_log = 1;
    o->pos_cape_neg_cin = 1;
    o->post_zero_cin = 0;
    o->metpy_compat = 141;
    o->exact_only = 0;
    o->mixed_layer_depth = 100.0;
    o->most_unstable_depth = 300.0;
}

xp_status xp_create(int device, xp_context **out_ctx) {
    if (!out_ctx) return fail(nullptr, XP_ERR_INVALID_ARGUMENT, "out_ctx is NULL");
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, XP_ERR_NO_DEVICE,
                    std::string("no CUDA device: ") + (e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e)));
    if (device < 0 || device >= count)
        return fail(nullptr, XP_ERR_INVALID_ARGUMENT, "device index out of range");
    xp_context *ctx = new xp_context();
    ctx->device = device;
    DeviceGuard guard(device);
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (const char *ev = getenv("XP_FAST_VOTE_MASK")) ctx->vote_mask = atoi(ev) & 15;
    {
        const unsigned hc = std::thread::hardware_concurrency();
        // staging copies of pageable caller arrays: half of the host's hardware threads, at most 16 (B200 box, 32
        // vCPUs, 3.1 M ERA5 columns through parcel_suite: 8 threads 65-68 ms per call, 16 threads 49-55, 24 threads 58-59)
        ctx->host_threads = (int)std::max(1u, std::min(16u, hc ? hc / 2 : 1u));
        if (const char *ev = getenv("XP_HOST_THREADS")) ctx->host_threads = std::max(1, std::min(64, atoi(ev)));
    }
    if (const char *ev = getenv("XP_HOST_BLOCK_MB")) {
        const int mb = atoi(ev);
        if (mb >= 1 && mb <= 4096) ctx->host_block_mb = mb;
    }
    if ((e = cudaMalloc(&ctx->d_flags, sizeof(uint32_t))) != cudaSuccess ||
        (e = cudaMemset(ctx->d_flags, 0, sizeof(uint32_t))) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev_mid)) != cudaSuccess) {
        g_create_error = std::string("xp_create: ") + cudaGetErrorString(e);
        delete ctx;
        return XP_ERR_CUDA;
    }
    *out_ctx = ctx;
    return XP_OK;
}

void xp_destroy(xp_context *ctx) {
    if (!ctx) return;
    {
        DeviceGuard guard(ctx->device);
        cudaFree(ctx->d_index);
        cudaFree(ctx->d_curves);
        cudaFree(ctx->d_flags);
        for (int s = 0; s < xp_context::kSlots; ++s) {
            if (ctx->slot_buf[s]) cudaFree(ctx->slot_buf[s]);
            if (ctx->slot_pin[s]) cudaFreeHost(ctx->slot_pin[s]);
            if (ctx->slot_stream[s]) cudaStreamDestroy(ctx->slot_stream[s]);
        }
        if (ctx->block_count_pin) cudaFreeHost(ctx->block_count_pin);
        for (auto &kv : ctx->scratch) cudaFree(kv.second.ptr);
        if (ctx->ev0) cudaEventDestroy(ctx->ev0);
        if (ctx->ev1) cudaEventDestroy(ctx->ev1);
        if (ctx->ev_mid) cudaEventDestroy(ctx->ev_mid);
    }
    delete ctx;
}

const char *xp_last_error(const xp_context *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

xp_status xp_take_flags(xp_context *ctx, void *stream, uint32_t *out_flags) {
    if (!ctx || !out_flags) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_CUDA(ctx, cudaMemcpyAsync(out_flags, ctx->d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    XP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, sizeof(uint32_t), st));
    XP_CUDA(ctx, cudaStreamSynchronize(st));
    return XP_OK;
}

static xp_status ensure_table_memory(xp_context *ctx) {
    if (!ctx->d_index) XP_CUDA(ctx, cudaMalloc(&ctx->d_index, (size_t)kNP * kNT * sizeof(uint16_t)));
    if (!ctx->d_curves) XP_CUDA(ctx, cudaMalloc(&ctx->d_curves, (size_t)kNAdiabats * kNP * sizeof(float)));
    return XP_OK;
}

xp_status xp_tables_build(xp_context *ctx, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DeviceGuard guard(ctx->device);
    xp_status st = ensure_table_memory(ctx);
    if (st != XP_OK) return st;
    uint32_t *scratch = nullptr;
    XP_CUDA(ctx, cudaMalloc(&scratch, (size_t)kNP * kNT * sizeof(uint32_t)));
    launch_build_tables(ctx->d_index, ctx->d_curves, scratch, (cudaStream_t)stream);
    ctx->launches += 2;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(scratch);
    XP_CUDA(ctx, e);
    ctx->tables = true;
    return XP_OK;
}

xp_status xp_tables_set(xp_context *ctx, const uint16_t *index_grid_host, const float *curves_host) {
    if (!ctx || !index_grid_host || !curves_host) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DeviceGuard guard(ctx->device);
    xp_status st = ensure_table_memory(ctx);
    if (st != XP_OK) return st;
    XP_CUDA(ctx, cudaMemcpy(ctx->d_index, index_grid_host, (size_t)kNP * kNT * sizeof(uint16_t), cudaMemcpyHostToDevice));
    XP_CUDA(ctx, cudaMemcpy(ctx->d_curves, curves_host, (size_t)kNAdiabats * kNP * sizeof(float), cudaMemcpyHostToDevice));
    ctx->tables = true;
    return XP_OK;
}

xp_status xp_tables_get(xp_context *ctx, uint16_t *index_grid_host, float *curves_host) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    DeviceGuard guard(ctx->device);
    if (index_grid_host)
        XP_CUDA(ctx, cudaMemcpy(index_grid_host, ctx->d_index, (size_t)kNP * kNT * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    if (curves_host)
        XP_CUDA(ctx, cudaMemcpy(curves_host, ctx->d_curves, (size_t)kNAdiabats * kNP * sizeof(float), cudaMemcpyDeviceToHost));
    return XP_OK;
}

int xp_tables_loaded(const xp_context *ctx) { return ctx && ctx->tables ? 1 : 0; }

xp_status xp_cape_cin(xp_context *ctx, const xp_columns *cols, int32_t kind,
                      const xp_parcel_in *explicit_parcel, const xp_options *opts,
                      const xp_parcel_out *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    if (kind < 0 || kind > 3) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "unknown parcel kind");
    if (!out) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "out is NULL");
    const xp_parcel_out *outs[4] = {nullptr, nullptr, nullptr, nullptr};
    outs[kind] = out;
    return run_any(ctx, cols, 1 << kind, outs, explicit_parcel, opts, stream);
}

xp_status xp_suite(xp_context *ctx, const xp_columns *cols, const xp_options *opts,
                   const xp_parcel_out *out_sb, const xp_parcel_out *out_ml,
                   const xp_parcel_out *out_mu, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    const xp_parcel_out *outs[4] = {out_sb, out_ml, out_mu, nullptr};
    int mask = (out_sb ? kSB : 0) | (out_ml ? kML : 0) | (out_mu ? kMU : 0);
    if (!mask) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "no outputs requested");
    return run_any(ctx, cols, mask, outs, nullptr, opts, stream);
}

#define XP_DISPATCH(dtype, CALL_F32, CALL_F64)                                  \
    do {                                                                        \
        if ((dtype) == XP_F32) { CALL_F32; }                                    \
        else if ((dtype) == XP_F64) { CALL_F64; }                               \
        else return fail(ctx, XP_ERR_INVALID_ARGUMENT, "dtype must be XP_F32 or XP_F64"); \
    } while (0)

xp_status xp_lcl(xp_context *ctx, const void *p, const void *t, const void *td, int64_t n,
                 int32_t dtype, const xp_options *opts, void *lcl_p, void *lcl_t, void *lcl_tv,
                 void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!p || !t || !td || n < 0) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad lcl arguments");
    DeviceGuard guard(ctx->device);
    const Opts o = to_opts(ctx, opts);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_lcl<float>((const float *)p, (const float *)t, (const float *)td, n, o, (float *)lcl_p, (float *)lcl_t, (float *)lcl_tv, st),
                launch_lcl<double>((const double *)p, (const double *)t, (const double *)td, n, o, (double *)lcl_p, (double *)lcl_t, (double *)lcl_tv, st));
    ctx->launches += n > 0;
    return check_cuda(ctx, cudaGetLastError(), "lcl kernel launch");
}

xp_status xp_moist_lapse(xp_context *ctx, const void *pressure, int64_t level_stride,
                         int32_t n_levels, int64_t n_columns, int32_t dtype,
                         const void *parcel_temperature, const void *parcel_pressure,
                         void *out_temperature, int64_t out_level_stride, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (!pressure || !parcel_temperature || !parcel_pressure || !out_temperature)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad moist_lapse arguments");
    DeviceGuard guard(ctx->device);
    Tables tb = {ctx->d_index, ctx->d_curves};
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_moist_lapse<float>((const float *)pressure, level_stride, n_levels, n_columns, tb, (const float *)parcel_temperature, (const float *)parcel_pressure, (float *)out_temperature, out_level_stride, st),
                launch_moist_lapse<double>((const double *)pressure, level_stride, n_levels, n_columns, tb, (const double *)parcel_temperature, (const double *)parcel_pressure, (double *)out_temperature, out_level_stride, st));
    ctx->launches += n_columns > 0;
    return check_cuda(ctx, cudaGetLastError(), "moist_lapse kernel launch");
}

xp_status xp_parcel_profile(xp_context *ctx, const void *pressure, int64_t level_stride,
                            int32_t n_levels, int64_t n_columns, int32_t dtype,
                            const xp_parcel_in *parcel, const xp_options *opts,
                            void *out_temperature, void *out_virtual_temperature,
                            int64_t out_level_stride, void *lcl_pressure, void *lcl_temperature,
                            void *lcl_virtual_temperature, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (!pressure || !parcel || !parcel->pressure || !parcel->temperature || !parcel->dewpoint)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad parcel_profile arguments");
    DeviceGuard guard(ctx->device);
    Tables tb = {ctx->d_index, ctx->d_curves};
    const Opts o = to_opts(ctx, opts);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == XP_F32) {
        ParcelArg<float> pa = {(const float *)parcel->pressure, (const float *)parcel->temperature, (const float *)parcel->dewpoint};
        launch_parcel_profile<float>((const float *)pressure, level_stride, n_levels, n_columns, tb, o, pa, (float *)out_temperature, (float *)out_virtual_temperature, out_level_stride, (float *)lcl_pressure, (float *)lcl_temperature, (float *)lcl_virtual_temperature, st);
    } else if (dtype == XP_F64) {
        ParcelArg<double> pa = {(const double *)parcel->pressure, (const double *)parcel->temperature, (const double *)parcel->dewpoint};
        launch_parcel_profile<double>((const double *)pressure, level_stride, n_levels, n_columns, tb, o, pa, (double *)out_temperature, (double *)out_virtual_temperature, out_level_stride, (double *)lcl_pressure, (double *)lcl_temperature, (double *)lcl_virtual_temperature, st);
    } else {
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "dtype must be XP_F32 or XP_F64");
    }
    ctx->launches += n_columns > 0;
    return check_cuda(ctx, cudaGetLastError(), "parcel_profile kernel launch");
}

xp_status xp_lfc_el(xp_context *ctx, const void *pressure, const void *parcel_temperature,
                    const void *temperature, int64_t level_stride, int32_t n_levels,
                    int64_t n_columns, int32_t dtype, const void *lcl_pressure,
                    const void *lcl_temperature, void *lfc_pressure, void *lfc_temperature,
                    void *el_pressure, void *el_temperature, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!pressure || !parcel_temperature || !temperature || !lcl_pressure || !lcl_temperature)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad lfc_el arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_lfc_el<float>((const float *)pressure, (const float *)parcel_temperature, (const float *)temperature, level_stride, n_levels, n_columns, (const float *)lcl_pressure, (const float *)lcl_temperature, (float *)lfc_pressure, (float *)lfc_temperature, (float *)el_pressure, (float *)el_temperature, ctx->d_flags, st),
                launch_lfc_el<double>((const double *)pressure, (const double *)parcel_temperature, (const double *)temperature, level_stride, n_levels, n_columns, (const double *)lcl_pressure, (const double *)lcl_temperature, (double *)lfc_pressure, (double *)lfc_temperature, (double *)el_pressure, (double *)el_temperature, ctx->d_flags, st));
    ctx->launches += n_columns > 0;
    return check_cuda(ctx, cudaGetLastError(), "lfc_el kernel launch");
}

xp_status xp_cape_cin_base(xp_context *ctx, const void *pressure, const void *temperature,
                           const void *parcel_temperature, int64_t level_stride,
                           int32_t n_levels, int64_t n_columns, int32_t dtype,
                           const void *lfc_pressure, const void *el_pressure,
                           const xp_options *opts, void *cape, void *cin, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!pressure || !temperature || !parcel_temperature || !lfc_pressure || !el_pressure)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad cape_cin_base arguments");
    DeviceGuard guard(ctx->device);
    const Opts o = to_opts(ctx, opts);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_cape_cin_base<float>((const float *)pressure, (const float *)temperature, (const float *)parcel_temperature, level_stride, n_levels, n_columns, (const float *)lfc_pressure, (const float *)el_pressure, o, (float *)cape, (float *)cin, st),
                launch_cape_cin_base<double>((const double *)pressure, (const double *)temperature, (const double *)parcel_temperature, level_stride, n_levels, n_columns, (const double *)lfc_pressure, (const double *)el_pressure, o, (double *)cape, (double *)cin, st));
    ctx->launches += n_columns > 0;
    return check_cuda(ctx, cudaGetLastError(), "cape_cin_base kernel launch");
}

xp_status xp_interp_levels(xp_context *ctx, const void *coords, int64_t coords_level_stride,
                           int32_t coords_is_1d, const void *const *fields, void *const *outputs,
                           int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                           int32_t dtype, const void *at, double at_scalar, int32_t log_coords,
                           void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!coords || !fields || !outputs || n_fields < 1 || n_fields > 4 || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad interp_levels arguments");
    for (int f = 0; f < n_fields; ++f)
        if (!fields[f] || !outputs[f]) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "interp_levels: NULL field/output");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_interp_levels<float>((const float *)coords, coords_level_stride, coords_is_1d, (const float *const *)fields, (float *const *)outputs, n_fields, level_stride, n_levels, n_columns, (const float *)at, at_scalar, log_coords, st),
                launch_interp_levels<double>((const double *)coords, coords_level_stride, coords_is_1d, (const double *const *)fields, (double *const *)outputs, n_fields, level_stride, n_levels, n_columns, (const double *)at, at_scalar, log_coords, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "interp_levels kernel launch");
}

xp_status xp_level_crossing(xp_context *ctx, const void *coords, int64_t coords_level_stride,
                            int32_t coords_is_1d, const void *field, int64_t level_stride,
                            int32_t n_levels, int64_t n_columns, int32_t dtype, double level,
                            void *output, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!coords || !field || !output || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad level_crossing arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_level_crossing<float>((const float *)coords, coords_level_stride, coords_is_1d, (const float *)field, level_stride, n_levels, n_columns, level, (float *)output, st),
                launch_level_crossing<double>((const double *)coords, coords_level_stride, coords_is_1d, (const double *)field, level_stride, n_levels, n_columns, level, (double *)output, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "level_crossing kernel launch");
}

xp_status xp_mixed_layer(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                         int32_t pressure_is_1d, const void *const *fields, void *const *outputs, int32_t n_fields,
                         int32_t pressure_field, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                         int32_t dtype, double depth, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!pressure || !fields || !outputs || n_fields < 1 || n_fields > 4 || pressure_field >= n_fields || n_levels < 1 ||
        n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad mixed_layer arguments");
    for (int f = 0; f < n_fields; ++f)
        if (!fields[f] || !outputs[f]) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "mixed_layer: NULL field/output");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_mixed_layer<float>((const float *)pressure, pressure_level_stride, pressure_is_1d, (const float *const *)fields, (float *const *)outputs, n_fields, pressure_field, level_stride, n_levels, n_columns, depth, st),
                launch_mixed_layer<double>((const double *)pressure, pressure_level_stride, pressure_is_1d, (const double *const *)fields, (double *const *)outputs, n_fields, pressure_field, level_stride, n_levels, n_columns, depth, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "mixed_layer kernel launch");
}

xp_status xp_mixed_parcel(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                          int32_t pressure_is_1d, const void *temperature, const void *dewpoint,
                          int64_t level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype, double depth,
                          const xp_mixed_parcel_out *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!pressure || !temperature || !dewpoint || !out || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad mixed_parcel arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    void *o6[6] = {out->theta, out->mixing_ratio, out->temperature, out->vapour_pressure, out->dewpoint, out->pressure};
    XP_DISPATCH(dtype,
                launch_mixed_parcel<float>((const float *)pressure, pressure_level_stride, pressure_is_1d, (const float *)temperature, (const float *)dewpoint, level_stride, n_levels, n_columns, depth, (float *const *)o6, st),
                launch_mixed_parcel<double>((const double *)pressure, pressure_level_stride, pressure_is_1d, (const double *)temperature, (const double *)dewpoint, level_stride, n_levels, n_columns, depth, (double *const *)o6, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "mixed_parcel kernel launch");
}

xp_status xp_layer_bounds(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                          int32_t pressure_is_1d, int32_t n_levels, int64_t n_columns, int32_t dtype, double depth,
                          int32_t interpolate, void *bottom_pressure, void *top_pressure, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!pressure || (!bottom_pressure && !top_pressure) || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad layer_bounds arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_layer_bounds<float>((const float *)pressure, pressure_level_stride, pressure_is_1d, n_levels, n_columns, depth, interpolate, (float *)bottom_pressure, (float *)top_pressure, st),
                launch_layer_bounds<double>((const double *)pressure, pressure_level_stride, pressure_is_1d, n_levels, n_columns, depth, interpolate, (double *)bottom_pressure, (double *)top_pressure, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "layer_bounds kernel launch");
}

xp_status xp_insert_level(xp_context *ctx, const void *coords, int64_t coords_level_stride, int32_t coords_is_1d,
                          const void *level_coord, const void *const *fields, const void *const *level_values,
                          void *const *outputs, int32_t n_fields, void *coords_out, int64_t level_stride,
                          int64_t out_level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!coords || !level_coord || n_fields < 0 || n_fields > 4 || (n_fields == 0 && !coords_out) ||
        (n_fields > 0 && (!fields || !level_values || !outputs)) || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad insert_level arguments");
    for (int f = 0; f < n_fields; ++f)
        if (!fields[f] || !level_values[f] || !outputs[f])
            return fail(ctx, XP_ERR_INVALID_ARGUMENT, "insert_level: NULL field/level/output");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_insert_level<float>((const float *)coords, coords_level_stride, coords_is_1d, (const float *)level_coord, (const float *const *)fields, (const float *const *)level_values, (float *const *)outputs, (float *)coords_out, n_fields, level_stride, out_level_stride, n_levels, n_columns, st),
                launch_insert_level<double>((const double *)coords, coords_level_stride, coords_is_1d, (const double *)level_coord, (const double *const *)fields, (const double *const *)level_values, (double *const *)outputs, (double *)coords_out, n_fields, level_stride, out_level_stride, n_levels, n_columns, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "insert_level kernel launch");
}

xp_status xp_shift_out_nans(xp_context *ctx, const void *ref_field, const void *const *fields, void *const *outputs,
                            int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                            int32_t dtype, int32_t *level_shift, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!ref_field || n_fields < 0 || n_fields > 4 || (n_fields == 0 && !level_shift) ||
        (n_fields > 0 && (!fields || !outputs)) || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad shift_out_nans arguments");
    for (int f = 0; f < n_fields; ++f)
        if (!fields[f] || !outputs[f] || fields[f] == outputs[f])
            return fail(ctx, XP_ERR_INVALID_ARGUMENT, "shift_out_nans: NULL or aliased field/output");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_shift_out_nans<float>((const float *)ref_field, (const float *const *)fields, (float *const *)outputs, n_fields, level_stride, n_levels, n_columns, level_shift, st),
                launch_shift_out_nans<double>((const double *)ref_field, (const double *const *)fields, (double *const *)outputs, n_fields, level_stride, n_levels, n_columns, level_shift, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "shift_out_nans kernel launch");
}

xp_status xp_trapz(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *const *fields,
                   void *const *outputs, int32_t n_fields, int64_t level_stride, int32_t n_levels, int64_t n_columns,
                   int32_t dtype, const uint8_t *mask, int64_t mask_level_stride, int32_t sign, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!x || !fields || !outputs || n_fields < 1 || n_fields > 4 || n_levels < 1 || n_columns < 0 || sign < -1 || sign > 1)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad trapz arguments");
    for (int f = 0; f < n_fields; ++f)
        if (!fields[f] || !outputs[f]) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "trapz: NULL field/output");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_trapz<float>((const float *)x, x_level_stride, x_is_1d, (const float *const *)fields, (float *const *)outputs, n_fields, level_stride, n_levels, n_columns, mask, mask_level_stride, sign, st),
                launch_trapz<double>((const double *)x, x_level_stride, x_is_1d, (const double *const *)fields, (double *const *)outputs, n_fields, level_stride, n_levels, n_columns, mask, mask_level_stride, sign, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "trapz kernel launch");
}

xp_status xp_find_intersections(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *a,
                                const void *b, int64_t level_stride, int64_t out_level_stride, int32_t n_levels,
                                int64_t n_columns, int32_t dtype, int32_t log_x, const xp_intersections_out *out,
                                void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!x || !a || !b || !out || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad find_intersections arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    void *o6[6] = {out->all_intersect_x, out->all_intersect_y, out->increasing_x, out->increasing_y,
                   out->decreasing_x, out->decreasing_y};
    XP_DISPATCH(dtype,
                launch_find_intersections<float>((const float *)x, x_level_stride, x_is_1d, (const float *)a, (const float *)b, level_stride, out_level_stride, n_levels, n_columns, log_x, (float *const *)o6, st),
                launch_find_intersections<double>((const double *)x, x_level_stride, x_is_1d, (const double *)a, (const double *)b, level_stride, out_level_stride, n_levels, n_columns, log_x, (double *const *)o6, st));
    ctx->launches += n_levels >= 2;
    return check_cuda(ctx, cudaGetLastError(), "find_intersections kernel launch");
}

xp_status xp_interp1d(xp_context *ctx, const void *at, const void *xp, int32_t xp_is_1d, const void *fp, void *out,
                      int64_t n_rows, int32_t m, int32_t n, int32_t dtype, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_rows == 0 || m == 0) return XP_OK;
    if (!at || !xp || !fp || !out || n_rows < 0 || m < 0 || n < 1)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad interp1d arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_interp1d<float>((const float *)at, (const float *)xp, (const float *)fp, (float *)out, n_rows, m, n, xp_is_1d, st),
                launch_interp1d<double>((const double *)at, (const double *)xp, (const double *)fp, (double *)out, n_rows, m, n, xp_is_1d, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "interp1d kernel launch");
}

xp_status xp_trap_around_zeros(xp_context *ctx, const void *x, int64_t x_level_stride, int32_t x_is_1d, const void *y,
                               int64_t level_stride, int64_t out_level_stride, int32_t n_levels, int64_t n_columns,
                               int32_t dtype, int32_t log_x, const xp_zero_areas_out *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!x || !y || !out || n_levels < 1 || n_columns < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad trap_around_zeros arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    void *o5[5] = {out->area, out->x, out->dx, out->x_from, out->x_to};
    XP_DISPATCH(dtype,
                launch_trap_around_zeros<float>((const float *)x, x_level_stride, x_is_1d, (const float *)y, level_stride, out_level_stride, n_levels, n_columns, log_x, (float *const *)o5, out->mask, st),
                launch_trap_around_zeros<double>((const double *)x, x_level_stride, x_is_1d, (const double *)y, level_stride, out_level_stride, n_levels, n_columns, log_x, (double *const *)o5, out->mask, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "trap_around_zeros kernel launch");
}

xp_status xp_valid_data(xp_context *ctx, const void *pressure, int64_t pressure_level_stride, int32_t pressure_is_1d,
                        int32_t n_levels, int64_t n_columns, int32_t dtype, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n_columns == 0) return XP_OK;
    if (!pressure || n_levels < 1 || n_columns < 0) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad valid_data arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = pressure_is_1d ? 1 : n_columns;
    XP_DISPATCH(dtype,
                launch_pressure_order<float>((const float *)pressure, pressure_level_stride, pressure_is_1d, n_levels, n, ctx->d_flags, st),
                launch_pressure_order<double>((const double *)pressure, pressure_level_stride, pressure_is_1d, n_levels, n, ctx->d_flags, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "valid_data kernel launch");
}

xp_status xp_dewpoint_from_specific_humidity(xp_context *ctx, const void *pressure, const void *temperature,
                                             const void *specific_humidity, int64_t n, int32_t dtype,
                                             int32_t metpy_compat, void *dewpoint, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!pressure || !temperature || !specific_humidity || !dewpoint || n < 0 || (metpy_compat != 141 && metpy_compat != 162))
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad dewpoint_from_specific_humidity arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_dewpoint_from_q<float>((const float *)pressure, (const float *)temperature, (const float *)specific_humidity, n, metpy_compat, (float *)dewpoint, st),
                launch_dewpoint_from_q<double>((const double *)pressure, (const double *)temperature, (const double *)specific_humidity, n, metpy_compat, (double *)dewpoint, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "dewpoint_from_specific_humidity kernel launch");
}

xp_status xp_saturation_mixing_ratio(xp_context *ctx, const void *pressure, const void *temperature, int64_t n,
                                     int32_t dtype, void *mixing_ratio, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!pressure || !temperature || !mixing_ratio || n < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad saturation_mixing_ratio arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_sat_mixing_ratio<float>((const float *)pressure, (const float *)temperature, n, (float *)mixing_ratio, st),
                launch_sat_mixing_ratio<double>((const double *)pressure, (const double *)temperature, n, (double *)mixing_ratio, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "saturation_mixing_ratio kernel launch");
}

xp_status xp_dry_lapse(xp_context *ctx, const void *pressure, const void *parcel_temperature,
                       const void *parcel_pressure, int64_t n, int32_t dtype, void *temperature, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!pressure || !parcel_temperature || !parcel_pressure || !temperature || n < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad dry_lapse arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_dry_lapse<float>((const float *)pressure, (const float *)parcel_temperature, (const float *)parcel_pressure, n, (float *)temperature, st),
                launch_dry_lapse<double>((const double *)pressure, (const double *)parcel_temperature, (const double *)parcel_pressure, n, (double *)temperature, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "dry_lapse kernel launch");
}

xp_status xp_mixing_ratio(xp_context *ctx, const void *temperature, const void *dewpoint, const void *pressure,
                          int64_t n, int32_t dtype, int32_t metpy_compat, void *mixing_ratio, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!temperature || !dewpoint || !pressure || !mixing_ratio || n < 0 || (metpy_compat != 141 && metpy_compat != 162))
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad mixing_ratio arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_mixing_ratio<float>((const float *)temperature, (const float *)dewpoint, (const float *)pressure, n, metpy_compat, (float *)mixing_ratio, st),
                launch_mixing_ratio<double>((const double *)temperature, (const double *)dewpoint, (const double *)pressure, n, metpy_compat, (double *)mixing_ratio, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "mixing_ratio kernel launch");
}

xp_status xp_virtual_temperature(xp_context *ctx, const void *temperature, const void *mixing_ratio, int64_t n,
                                 int32_t dtype, double epsilon, void *virtual_temperature, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!temperature || !mixing_ratio || !virtual_temperature || n < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad virtual_temperature arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_virtual_temperature<float>((const float *)temperature, (const float *)mixing_ratio, n, epsilon, (float *)virtual_temperature, st),
                launch_virtual_temperature<double>((const double *)temperature, (const double *)mixing_ratio, n, epsilon, (double *)virtual_temperature, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "virtual_temperature kernel launch");
}

xp_status xp_wet_bulb_temperature(xp_context *ctx, const void *pressure, const void *temperature,
                                  const void *dewpoint, int64_t n, int32_t dtype, void *wet_bulb, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (n == 0) return XP_OK;
    if (!pressure || !temperature || !dewpoint || !wet_bulb || n < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad wet_bulb_temperature arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const Tables tb = {ctx->d_index, ctx->d_curves};
    XP_DISPATCH(dtype,
                launch_wet_bulb<float>((const float *)pressure, (const float *)temperature, (const float *)dewpoint, n, tb, (float *)wet_bulb, st),
                launch_wet_bulb<double>((const double *)pressure, (const double *)temperature, (const double *)dewpoint, n, tb, (double *)wet_bulb, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "wet_bulb_temperature kernel launch");
}

// Downdraft CAPE, contract in include/xparcel.h and xp_downdraft.cuh (DESIGN.md section 3.12).
xp_status xp_downdraft_cape(xp_context *ctx, const void *pressure, int64_t pressure_level_stride,
                            int32_t pressure_is_1d, const void *temperature, const void *dewpoint,
                            int64_t level_stride, int32_t n_levels, int64_t n_columns, int32_t dtype,
                            int32_t metpy_compat, const xp_downdraft_out *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (n_columns == 0) return XP_OK;
    if (!pressure || !temperature || !dewpoint || !out || n_levels < 1 || n_columns < 0 ||
        (metpy_compat != 141 && metpy_compat != 162))
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad downdraft_cape arguments");
    if (n_levels > 1 && (level_stride < n_columns ||
                         pressure_level_stride < (pressure_is_1d ? 1 : n_columns) ||
                         (out->parcel_temperature && out->parcel_level_stride < n_columns)))
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "downdraft_cape: level strides smaller than a level");
    if (!out->dcape && !out->start_pressure && !out->start_temperature && !out->parcel_temperature) return XP_OK;
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const Tables tb = {ctx->d_index, ctx->d_curves};
    XP_DISPATCH(dtype,
                launch_downdraft_cape<float>((const float *)pressure, pressure_level_stride, pressure_is_1d, (const float *)temperature, (const float *)dewpoint, level_stride, n_levels, n_columns, metpy_compat, tb, (float *)out->dcape, (float *)out->start_pressure, (float *)out->start_temperature, (float *)out->parcel_temperature, out->parcel_level_stride, st),
                launch_downdraft_cape<double>((const double *)pressure, pressure_level_stride, pressure_is_1d, (const double *)temperature, (const double *)dewpoint, level_stride, n_levels, n_columns, metpy_compat, tb, (double *)out->dcape, (double *)out->start_pressure, (double *)out->start_temperature, (double *)out->parcel_temperature, out->parcel_level_stride, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "downdraft_cape kernel launch");
}

// Effective inflow layer, contract in include/xparcel.h and xp_effective.cuh (DESIGN.md section 3.13).
xp_status xp_effective_inflow_layer(xp_context *ctx, const xp_columns *cols, const xp_options *opts, double min_cape,
                                    double min_cin, const xp_effective_out *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    xp_status st = validate_cols(ctx, cols);
    if (st != XP_OK) return st;
    if (!out) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "out is NULL");
    if (cols->mem != XP_MEM_DEVICE)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "effective_inflow_layer: device memory only (mem = XP_MEM_DEVICE)");
    if (cols->dewpoint_is_specific_humidity)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "effective_inflow_layer: dewpoint_is_specific_humidity is not supported");
    if (cols->reserved_ != 0) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "reserved_ must be 0");
    if (!ctx->tables) return fail(ctx, XP_ERR_TABLES_NOT_LOADED, "Call load_moist_adiabat_lookups first.");
    if (cols->n_columns == 0) return XP_OK;
    if ((out->level_cape || out->level_cin) && out->level_out_stride < cols->n_columns)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "effective_inflow_layer: level_out_stride must be >= n_columns");
    if (cols->n_columns > (int64_t)1 << 40)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "effective_inflow_layer: more than 2^40 columns");
    if (!out->base_pressure && !out->top_pressure && !out->level_cape && !out->level_cin) return XP_OK;
    DeviceGuard guard(ctx->device);
    cudaStream_t s = (cudaStream_t)stream;
    const Opts o = to_opts(ctx, opts);
    void *scratch = nullptr;
    XP_CUDA(ctx, stream_scratch(ctx, s, effective_scratch_bytes(cols->n_columns), &scratch));
    if (ctx->last_fast_stream == s) ctx->last_was_fast = false;     // its fix-up list count is gone with the scratch
    const Tables tb = {ctx->d_index, ctx->d_curves};
    int rc;
    if (cols->dtype == XP_F32)
        rc = launch_effective<float>(to_cols<float>(cols, o), tb, o, min_cape, min_cin, (float *)out->base_pressure,
                                     (float *)out->top_pressure, (float *)out->level_cape, (float *)out->level_cin,
                                     out->level_out_stride, ctx->d_flags, scratch, ctx->sm_count, s);
    else
        rc = launch_effective<double>(to_cols<double>(cols, o), tb, o, min_cape, min_cin, (double *)out->base_pressure,
                                      (double *)out->top_pressure, (double *)out->level_cape, (double *)out->level_cin,
                                      out->level_out_stride, ctx->d_flags, scratch, ctx->sm_count, s);
    if (rc < 0) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "effective_inflow_layer: too many levels on a shared axis");
    ctx->launches += 2;
    return check_cuda(ctx, cudaGetLastError(), "effective_inflow_layer kernel launch");
}

xp_status xp_significant_hail_parameter(xp_context *ctx, const void *mucape, const void *mixing_ratio,
                                        const void *lapse, const void *temp_500, const void *shear,
                                        const void *flh, int64_t n, int32_t dtype, void *ship, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!mucape || !mixing_ratio || !lapse || !temp_500 || !shear || !flh || !ship || n < 0)
        return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad significant_hail_parameter arguments");
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    const void *in[6] = {mucape, mixing_ratio, lapse, temp_500, shear, flh};
    XP_DISPATCH(dtype,
                launch_ship<float>((const float *const *)in, n, (float *)ship, st),
                launch_ship<double>((const double *const *)in, n, (double *)ship, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "significant_hail_parameter kernel launch");
}

xp_status xp_storm_proxies(xp_context *ctx, const xp_proxy_inputs *in, int64_t n, int32_t dtype,
                           const xp_proxy_outputs *out, void *stream) {
    if (!ctx) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return XP_OK;
    if (!in || !out || n < 0) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "bad storm_proxies arguments");
    const void *iv[13] = {in->mixed_100_cape, in->mixed_50_cape, in->mu_cape, in->shear_magnitude,
                          in->mixed_100_lifted_index, in->mixed_100_dci, in->positive_shear, in->mixed_50_cin,
                          in->mixed_100_cin, in->lapse_rate_700_500, in->mu_mixing_ratio, in->temp_500,
                          in->freezing_level};
    for (int k = 0; k < 13; ++k)
        if (!iv[k]) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "storm_proxies: NULL input");
    uint8_t *fl[9] = {out->craven2004, out->kunz2007, out->trapp2007, out->marsh2009, out->allen2011,
                      out->allen2014, out->eccel2012, out->mohr2013, out->ship_0_1};
    DeviceGuard guard(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    XP_DISPATCH(dtype,
                launch_storm_proxies<float>((const float *const *)iv, fl, (float *)out->ship, n, st),
                launch_storm_proxies<double>((const double *const *)iv, fl, (double *)out->ship, n, st));
    ctx->launches += 1;
    return check_cuda(ctx, cudaGetLastError(), "storm_proxies kernel launch");
}

uint64_t xp_launch_count(const xp_context *ctx) { return ctx ? ctx->launches : 0; }

xp_status xp_last_exact_count(xp_context *ctx, int64_t *out_count) {
    if (!ctx || !out_count) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    *out_count = -1;
    if (ctx->last_was_host) { *out_count = ctx->last_host_exact; return XP_OK; }    // every block of the call
    if (!ctx->last_was_fast) return XP_OK;
    DeviceGuard guard(ctx->device);
    auto it = ctx->scratch.find(ctx->last_fast_stream);
    if (it == ctx->scratch.end() || !it->second.ptr) return XP_OK;
    *out_count = (int64_t)fast_last_list_count(it->second.ptr, ctx->last_fast_stream);
    return check_cuda(ctx, cudaGetLastError(), "xp_last_exact_count");
}

xp_status xp_last_kernel_ms(xp_context *ctx, float *out_ms) {
    if (!ctx || !out_ms) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->ev_valid) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "no timed launch yet");
    DeviceGuard guard(ctx->device);
    XP_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    XP_CUDA(ctx, cudaEventElapsedTime(out_ms, ctx->ev0, ctx->ev1));
    return XP_OK;
}

xp_status xp_last_kernel_split_ms(xp_context *ctx, float *out_sweep_ms, float *out_fixup_ms) {
    if (!ctx || !out_sweep_ms || !out_fixup_ms) return XP_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->ev_valid || !ctx->ev_split) return fail(ctx, XP_ERR_INVALID_ARGUMENT, "no timed fast-path launch yet");
    DeviceGuard guard(ctx->device);
    XP_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    XP_CUDA(ctx, cudaEventElapsedTime(out_sweep_ms, ctx->ev0, ctx->ev_mid));
    XP_CUDA(ctx, cudaEventElapsedTime(out_fixup_ms, ctx->ev_mid, ctx->ev1));
    return XP_OK;
}

}  // extern "C"
