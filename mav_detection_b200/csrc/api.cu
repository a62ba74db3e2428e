// C ABI of libmavd (include/mavd.h): handle lifecycle, parameter tables, stage entry points and the
// whole-path calls.  No exceptions cross this boundary; every failure is an int status plus a
// thread-local message.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"

namespace mavd {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int alloc_slot(mavd_handle h, mavd_handle_s::HostSlot& S) {
    Arena& A = h->arena;
    const int F = h->max_frames, B = h->cfg.max_pairs;
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    int rc;
    if ((rc = A.alloc(&S.d_frames, (size_t)F * npx)) != MAVD_OK) return rc;
    if ((rc = A.alloc(&S.d_samples, (size_t)B * MAVD_SAMPLES_PER_FRAME)) != MAVD_OK) return rc;
    if ((rc = A.alloc(&S.d_sky, B * npx)) != MAVD_OK) return rc;
    if ((rc = A.alloc(&S.d_seg, B * npx)) != MAVD_OK) return rc;
    if ((rc = A.alloc(&S.d_records, (size_t)B)) != MAVD_OK) return rc;
    if ((rc = A.alloc(&S.d_fixed, B * npx)) != MAVD_OK) return rc;
    MAVD_CUDA(cudaEventCreateWithFlags(&S.ev_in, cudaEventDisableTiming));
    MAVD_CUDA(cudaEventCreateWithFlags(&S.ev_done, cudaEventDisableTiming));
    MAVD_CUDA(cudaEventCreateWithFlags(&S.ev_out, cudaEventDisableTiming));
    return MAVD_OK;
}

}  // namespace mavd

using namespace mavd;

static void drop_graphs(mavd_handle h);

// device memory, streams, events, graphs and pinned staging of a handle, then the handle
static void release(mavd_handle H) {
    for (void* p : H->arena.ptrs) cudaFree(p);
    drop_graphs(H);
    for (auto& S : H->slot) {
        if (S.ev_in) cudaEventDestroy(S.ev_in);
        if (S.ev_done) cudaEventDestroy(S.ev_done);
        if (S.ev_out) cudaEventDestroy(S.ev_out);
    }
    if (H->s_aux) cudaStreamDestroy(H->s_aux);
    if (H->ev_fork) cudaEventDestroy(H->ev_fork);
    if (H->ev_join) cudaEventDestroy(H->ev_join);
    if (H->ev_pyr) cudaEventDestroy(H->ev_pyr);
    if (H->s_in) cudaStreamDestroy(H->s_in);
    if (H->s_out) cudaStreamDestroy(H->s_out);
    if (H->s_main) cudaStreamDestroy(H->s_main);
    if (H->ev_main_in) cudaEventDestroy(H->ev_main_in);
    if (H->ev_main_out) cudaEventDestroy(H->ev_main_out);
    for (cudaEvent_t e : H->imu_ev)
        if (e) cudaEventDestroy(e);
    if (H->h_imu_ring) cudaFreeHost(H->h_imu_ring);
    for (cudaEvent_t e : H->stream_ev)
        if (e) cudaEventDestroy(e);
    if (H->h_stream_ring) cudaFreeHost(H->h_stream_ring);
    for (auto& r : H->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (cudaEvent_t e : H->prof.pool) cudaEventDestroy(e);
    delete H;
}

#define TRY(x)                       \
    do {                             \
        int rc__ = (x);              \
        if (rc__ != MAVD_OK) return rc__; \
    } while (0)

extern "C" {

int mavd_abi_version(void) { return MAVD_ABI_VERSION; }
const char* mavd_last_error(void) { return g_err; }
int64_t mavd_launch_count(void) { return g_launches.load(); }

void mavd_default_detect_params(mavd_detect_params* p) {
    if (!p) return;
    p->magnitude_threshold = 2.5;  // focus_of_expansion.py:22
    p->ransac_threshold = 30.0;    // focus_of_expansion.py:23
    p->dyn_offset = 0.25;          // processor.py:334-335
    p->dyn_base = 0.5;
    p->dyn_gain = 8.0;
    p->dyn_min_mag = 0.5;          // processor.py:338
    p->fixed_min_mag = 1.0;        // processor.py:341
    p->fixed_angle = 15.0;         // processor.py:340
}

static int validate(const mavd_config* c) {
    MAVD_REQUIRE(c != nullptr, MAVD_ERR_INVALID, "config is NULL");
    const mavd_farneback_params& f = c->farneback;
    MAVD_REQUIRE(c->width >= 8 && c->height >= 8 && c->width <= 16384 && c->height <= 16384, MAVD_ERR_INVALID,
                 "frame size %dx%d out of range", c->width, c->height);
    MAVD_REQUIRE(c->max_pairs >= 1, MAVD_ERR_INVALID, "max_pairs must be >= 1");
    MAVD_REQUIRE(f.pyr_scale > 0.0 && f.pyr_scale < 1.0, MAVD_ERR_INVALID, "pyr_scale must be in (0, 1)");
    MAVD_REQUIRE(f.levels >= 0, MAVD_ERR_INVALID, "levels must be >= 0");
    MAVD_REQUIRE(f.iterations >= 1, MAVD_ERR_UNSUPPORTED, "iterations must be >= 1");
    MAVD_REQUIRE(f.winsize >= 2 && f.winsize / 2 <= kMaxWinHalf, MAVD_ERR_UNSUPPORTED,
                 "winsize %d unsupported (2..%d)", f.winsize, 2 * kMaxWinHalf + 1);
    MAVD_REQUIRE(f.poly_n >= 1 && f.poly_n <= kMaxPolyN, MAVD_ERR_UNSUPPORTED, "poly_n %d unsupported (1..%d)",
                 f.poly_n, kMaxPolyN);
    MAVD_REQUIRE((f.flags & ~MAVD_FARNEBACK_GAUSSIAN) == 0, MAVD_ERR_UNSUPPORTED,
                 "flags 0x%x unsupported (only OPTFLOW_FARNEBACK_GAUSSIAN)", f.flags);
    return MAVD_OK;
}

int mavd_create(const mavd_config* cfg, mavd_handle* out) {
    MAVD_REQUIRE(out != nullptr, MAVD_ERR_INVALID, "out is NULL");
    *out = nullptr;
    TRY(validate(cfg));
    int ndev = 0;
    MAVD_CUDA(cudaGetDeviceCount(&ndev));
    MAVD_REQUIRE(cfg->device >= 0 && cfg->device < ndev, MAVD_ERR_CUDA, "CUDA device %d not available (%d devices)",
                 cfg->device, ndev);
    DeviceGuard dg(cfg->device);
    mavd_handle H = new (std::nothrow) mavd_handle_s();
    MAVD_REQUIRE(H != nullptr, MAVD_ERR_NOMEM, "out of host memory");
    H->cfg = *cfg;
    mavd_default_tuning(&H->tune);
    H->max_frames = 2 * cfg->max_pairs;  // worst case: independent pairs
    H->stream_live.assign(cfg->max_pairs, 0);
    H->stream_parity.assign(cfg->max_pairs, 0);
    int rc = MAVD_OK;
#define C_TRY(x) do { rc = (x); if (rc != MAVD_OK) { release(H); return rc; } } while (0)
    C_TRY(farneback_setup(H));
    C_TRY(detect_setup(H));
    // slot 0 is always there (mavd_detect_host stages through it); further slots appear on their first submit
    C_TRY(alloc_slot(H, H->slot[0]));
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&H->s_aux, cudaStreamNonBlocking, hi) != cudaSuccess ||
            cudaEventCreateWithFlags(&H->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&H->ev_join, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&H->ev_pyr, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            H->s_aux = nullptr;   // the path still works, just without the overlap
        }
        if (cudaStreamCreateWithFlags(&H->s_main, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&H->ev_main_in, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&H->ev_main_out, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            H->s_main = nullptr;  // default-stream calls then launch directly (no graph replay)
        }
    }
    {
        cudaError_t e = cudaMallocHost((void**)&H->h_imu_ring,
                                       sizeof(mavd_imu) * mavd_handle_s::kImuRing * (size_t)cfg->max_pairs);
        for (int k = 0; e == cudaSuccess && k < mavd_handle_s::kImuRing; ++k)
            e = cudaEventCreateWithFlags(&H->imu_ev[k], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            set_error("imu staging: %s", cudaGetErrorString(e));
            C_TRY(e == cudaErrorMemoryAllocation ? MAVD_ERR_NOMEM : MAVD_ERR_CUDA);
        }
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error("device error during create: %s", cudaGetErrorString(e));
        C_TRY(MAVD_ERR_CUDA);
    }
#undef C_TRY
    *out = H;
    return MAVD_OK;
}

int mavd_destroy(mavd_handle h) {
    if (!h) return MAVD_OK;
    DeviceGuard dg(h->cfg.device);
    cudaDeviceSynchronize();
    release(h);
    return MAVD_OK;
}

void mavd_default_tuning(mavd_tuning* t) {
    if (!t) return;
    memset(t, 0, sizeof(*t));
    t->mat_coord = 0;
    t->pyr_staged = 1;
    t->use_graph = 1;
    t->polyexp_tma = 1;
    t->iter_small_tiles = 1;
    t->use_pdl = 1;
    t->pyr_sweep = 1;
}

int mavd_set_tuning(mavd_handle h, const mavd_tuning* t) {
    MAVD_REQUIRE(h && t, MAVD_ERR_INVALID, "set_tuning: NULL argument");
    MAVD_REQUIRE(t->mat_coord >= 0 && t->mat_coord <= 2, MAVD_ERR_INVALID, "set_tuning: value out of range");
    DeviceGuard dg(h->cfg.device);
    MAVD_CUDA(cudaDeviceSynchronize());
    drop_graphs(h);
    h->tune = *t;
    return MAVD_OK;
}

int mavd_graph_stats(mavd_handle h, int32_t* n_captured, int32_t* n_direct) {
    MAVD_REQUIRE(h && n_captured && n_direct, MAVD_ERR_INVALID, "graph_stats: NULL argument");
    *n_captured = *n_direct = 0;
    for (const auto& g : h->graphs) ++*(g.exec ? n_captured : n_direct);
    return MAVD_OK;
}

int mavd_get_tuning(mavd_handle h, mavd_tuning* out) {
    MAVD_REQUIRE(h && out, MAVD_ERR_INVALID, "get_tuning: NULL argument");
    *out = h->tune;
    return MAVD_OK;
}

int mavd_profile_enable(mavd_handle h, int32_t on) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "profile: handle is NULL");
    DeviceGuard dg(h->cfg.device);
    MAVD_CUDA(cudaDeviceSynchronize());
    for (auto& r : h->prof.recs) { h->prof.pool.push_back(r.a); h->prof.pool.push_back(r.b); }
    h->prof.recs.clear();
    h->prof.on = on != 0;
    return MAVD_OK;
}

int mavd_profile_read(mavd_handle h, mavd_profile* out) {
    MAVD_REQUIRE(h && out, MAVD_ERR_INVALID, "profile: NULL argument");
    memset(out, 0, sizeof(*out));
    DeviceGuard dg(h->cfg.device);
    for (auto& r : h->prof.recs) {
        MAVD_CUDA(cudaEventSynchronize(r.b));
        float ms = 0.f;
        MAVD_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
        if (r.cls >= 0 && r.cls < MAVD_PROF_CLASSES) { out->ms[r.cls] += ms; out->launches[r.cls] += 1; }
        h->prof.pool.push_back(r.a);
        h->prof.pool.push_back(r.b);
    }
    h->prof.recs.clear();
    return MAVD_OK;
}

int mavd_profile_timeline(mavd_handle h, double* out, int32_t max_records, int32_t* n_out) {
    MAVD_REQUIRE(h && out && n_out, MAVD_ERR_INVALID, "profile_timeline: NULL argument");
    DeviceGuard dg(h->cfg.device);
    int n = 0;
    if (!h->prof.recs.empty()) {
        cudaEvent_t base = h->prof.recs[0].a;
        for (auto& r : h->prof.recs) {
            if (n >= max_records) break;
            MAVD_CUDA(cudaEventSynchronize(r.b));
            float t0 = 0.f, t1 = 0.f;
            MAVD_CUDA(cudaEventElapsedTime(&t0, base, r.a));
            MAVD_CUDA(cudaEventElapsedTime(&t1, base, r.b));
            out[3 * n] = r.cls; out[3 * n + 1] = t0; out[3 * n + 2] = t1;
            ++n;
        }
    }
    *n_out = n;
    return MAVD_OK;
}

int mavd_debug_force_generic_iteration(mavd_handle h, int32_t on) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "handle is NULL");
    DeviceGuard dg(h->cfg.device);
    MAVD_CUDA(cudaDeviceSynchronize());
    drop_graphs(h);                    // the flag changes the launch sequence
    h->force_generic_iter = on != 0;
    return MAVD_OK;
}

int mavd_workspace_bytes(mavd_handle h, size_t* out) {
    MAVD_REQUIRE(h && out, MAVD_ERR_INVALID, "NULL argument");
    *out = h->arena.bytes;
    return MAVD_OK;
}

int mavd_level_info(mavd_handle h, int32_t* n_images, int32_t* widths, int32_t* heights) {
    MAVD_REQUIRE(h && n_images, MAVD_ERR_INVALID, "NULL argument");
    *n_images = h->n_levels;
    for (int i = 0; i < h->n_levels; ++i) {
        if (widths) widths[i] = h->lv[i].w;
        if (heights) heights[i] = h->lv[i].h;
    }
    return MAVD_OK;
}

int mavd_bgr2gray(const uint8_t* d_bgr, uint8_t* d_gray, int64_t n_pixels, void* stream) {
    MAVD_REQUIRE(d_bgr && d_gray && n_pixels >= 0, MAVD_ERR_INVALID, "bgr2gray: bad arguments");
    if (n_pixels == 0) return MAVD_OK;
    return bgr2gray_run(d_bgr, d_gray, n_pixels, (cudaStream_t)stream);
}

static int check_batch(mavd_handle h, int n, const char* what) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "%s: handle is NULL", what);
    pdl_break(h, 0);        // the first kernel of a call is never chained to whatever ran before it on the stream
    pdl_break(h, 1);
    MAVD_REQUIRE(n >= 0 && n <= h->cfg.max_pairs, MAVD_ERR_INVALID, "%s: batch %d exceeds max_pairs %d", what, n,
                 h->cfg.max_pairs);
    return MAVD_OK;
}

// taps read "the last mavd_farneback call": recorded here, outside the (possibly replayed) launch sequence.  A
// non-stream call expands its frames into the R slots the streams keep theirs in: it ends every stream.
static void note_farneback_call(mavd_handle h, const uint8_t* d_frames, int n_pairs, int pair_stride, float* d_flow) {
    h->last_pairs = n_pairs;
    h->last_stride = pair_stride;
    h->last_flow0 = d_flow;
    h->last_frames = d_frames;
    h->last_was_stream = false;
    std::fill(h->stream_live.begin(), h->stream_live.end(), 0);
}

int mavd_farneback_tap(mavd_handle h, int32_t kind, int32_t level, int32_t index, float* d_out, void* stream) {
    MAVD_REQUIRE(h && d_out, MAVD_ERR_INVALID, "tap: NULL argument");
    DeviceGuard dg(h->cfg.device);
    MAVD_REQUIRE(!h->last_was_stream, MAVD_ERR_INVALID, "tap: the last Farneback call was a frame-stream call");
    MAVD_REQUIRE(index >= 0 && index < h->max_frames, MAVD_ERR_INVALID, "tap: index out of range");
    return farneback_tap(h, kind, level, index, d_out, (cudaStream_t)stream);
}

// ids of a frame-stream call: n distinct streams in 0..max_pairs-1; a step (not a start) also needs every one of them
// started and not ended since.  Checked before anything is staged or launched: a rejected call changes no stream.
static int check_stream_ids(mavd_handle h, const int32_t* h_ids, int n, bool step, const char* what) {
    MAVD_REQUIRE(h_ids != nullptr, MAVD_ERR_INVALID, "%s: ids array is NULL", what);
    std::vector<uint8_t> seen(h->cfg.max_pairs, 0);
    for (int i = 0; i < n; ++i) {
        const int32_t id = h_ids[i];
        MAVD_REQUIRE(id >= 0 && id < h->cfg.max_pairs, MAVD_ERR_INVALID, "%s: ids[%d] = %d outside 0..%d", what, i, id,
                     h->cfg.max_pairs - 1);
        MAVD_REQUIRE(!seen[id], MAVD_ERR_INVALID, "%s: stream %d appears twice", what, id);
        seen[id] = 1;
        MAVD_REQUIRE(!step || h->stream_live[id], MAVD_ERR_INVALID,
                     "%s: stream %d is not started (never, or ended by a non-stream Farneback call since)", what, id);
    }
    return MAVD_OK;
}

// The R slot tables of a checked stream call (FrameSlots), staged like the imu: a pinned ring slot, then an
// asynchronous copy into the fixed device tables that the (possibly replayed) launch sequence reads.  Frame i goes to
// the slot of its stream that does not hold the kept frame; pair i reads (kept, new).
static int upload_stream_slots(mavd_handle h, const int32_t* h_ids, int n, cudaStream_t s) {
    const int B = h->cfg.max_pairs;
    if (!h->d_stream_slots) TRY(h->arena.alloc(&h->d_stream_slots, (size_t)3 * B));
    for (cudaEvent_t& e : h->stream_ev)
        if (!e) MAVD_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (!h->h_stream_ring)
        MAVD_CUDA(cudaMallocHost((void**)&h->h_stream_ring, sizeof(int32_t) * 3 * B * mavd_handle_s::kImuRing));
    const int k = h->stream_next;
    h->stream_next = (k + 1) % mavd_handle_s::kImuRing;
    MAVD_CUDA(cudaEventSynchronize(h->stream_ev[k]));
    int32_t* stage = h->h_stream_ring + (size_t)k * 3 * B;
    for (int i = 0; i < n; ++i) {
        const int kept = 2 * h_ids[i] + h->stream_parity[h_ids[i]];
        stage[i] = kept ^ 1;
        stage[B + 2 * i] = kept;
        stage[B + 2 * i + 1] = kept ^ 1;
    }
    MAVD_CUDA(cudaMemcpyAsync(h->d_stream_slots, stage, sizeof(int32_t) * 3 * B, cudaMemcpyHostToDevice, s));
    MAVD_CUDA(cudaEventRecord(h->stream_ev[k], s));
    return MAVD_OK;
}

// a stream call was enqueued: each named stream now keeps the frame it was given
static void advance_streams(mavd_handle h, const int32_t* h_ids, int n) {
    for (int i = 0; i < n; ++i) {
        h->stream_parity[h_ids[i]] ^= 1;
        h->stream_live[h_ids[i]] = 1;
    }
    h->last_was_stream = true;
}

static int upload_imu(mavd_handle h, const mavd_imu* h_imu, int n, cudaStream_t s, int* n64, int* n32) {
    MAVD_REQUIRE(h_imu != nullptr, MAVD_ERR_INVALID, "imu array is NULL");
    int a = 0, b = 0, rot = 0;
    for (int i = 0; i < n; ++i) {
        if (h_imu[i].derotate) {
            MAVD_REQUIRE(h_imu[i].dt != 0.0, MAVD_ERR_INVALID, "imu[%d].dt is zero", i);
            ++a;
            // anything but an exact zero rotation (NaN included) takes the float64 derotation on the device
            if (!(h_imu[i].ang[0] == 0.0 && h_imu[i].ang[1] == 0.0 && h_imu[i].ang[2] == 0.0)) ++rot;
        } else {
            ++b;
        }
    }
    if (n64) *n64 = a;
    if (n32) *n32 = b;
    h->batch_rot = rot;
    // the caller's array is not retained: it is copied into the next pinned ring slot, and the asynchronous upload
    // reads that slot (a slot is rewritten only after the upload that used it has completed)
    const int k = h->imu_next;
    h->imu_next = (k + 1) % mavd_handle_s::kImuRing;
    MAVD_CUDA(cudaEventSynchronize(h->imu_ev[k]));
    mavd_imu* stage = h->h_imu_ring + (size_t)k * h->cfg.max_pairs;
    memcpy(stage, h_imu, sizeof(mavd_imu) * n);
    MAVD_CUDA(cudaMemcpyAsync(h->d_imu, stage, sizeof(mavd_imu) * n, cudaMemcpyHostToDevice, s));
    MAVD_CUDA(cudaEventRecord(h->imu_ev[k], s));
    return MAVD_OK;
}

int mavd_derotate(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, double* d_out, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "derotate"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_out, MAVD_ERR_INVALID, "derotate: NULL buffer");
    TRY(upload_imu(h, h_imu, n, (cudaStream_t)stream, nullptr, nullptr));
    return derotate_run(h, d_flow, 0, n, h->d_imu, d_out, (cudaStream_t)stream);
}

int mavd_derotate_f64(mavd_handle h, const double* d_flow, int32_t n, const mavd_imu* h_imu, double* d_out, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "derotate_f64"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_out, MAVD_ERR_INVALID, "derotate_f64: NULL buffer");
    TRY(upload_imu(h, h_imu, n, (cudaStream_t)stream, nullptr, nullptr));
    return derotate_run(h, d_flow, 1, n, h->d_imu, d_out, (cudaStream_t)stream);
}

int mavd_foe(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
             const int32_t* d_samples, double* d_foe, int32_t* d_n_intersections, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "foe"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_samples && d_foe, MAVD_ERR_INVALID, "foe: NULL buffer");
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    TRY(upload_imu(h, h_imu, n, (cudaStream_t)stream, nullptr, nullptr));
    return foe_run(h, d_flow, 0, n, h->d_imu, p, d_samples, d_foe, d_n_intersections ? d_n_intersections : h->d_ninter,
                   (cudaStream_t)stream);
}

int mavd_foe_dense(mavd_handle h, const void* d_flow, int32_t flow_is_f64, int32_t n, const mavd_detect_params* prm,
                   const int32_t* d_samples, double* d_foe, int32_t* d_n_intersections, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "foe_dense"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_samples && d_foe, MAVD_ERR_INVALID, "foe_dense: NULL buffer");
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    return foe_run(h, d_flow, flow_is_f64 ? 2 : 1, n, nullptr, p, d_samples, d_foe,
                   d_n_intersections ? d_n_intersections : h->d_ninter, (cudaStream_t)stream);
}

int mavd_ransac(mavd_handle h, const double* d_estimates, int32_t k, double ransac_threshold, double* d_foe,
                void* stream) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "ransac: handle is NULL");
    MAVD_REQUIRE(k >= 0 && d_foe && (k == 0 || d_estimates), MAVD_ERR_INVALID, "ransac: bad arguments");
    DeviceGuard dg(h->cfg.device);
    return ransac_run(d_estimates, k, ransac_threshold, d_foe, (cudaStream_t)stream);
}

int mavd_get_phi(mavd_handle h, const void* d_flow, int32_t flow_is_f64, int32_t n, const double* d_foe, void* d_phi,
                 double* d_max_phi, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "get_phi"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_foe && d_phi, MAVD_ERR_INVALID, "get_phi: NULL buffer");
    mavd_detect_params p;
    mavd_default_detect_params(&p);
    TRY(residual_run(h, d_flow, flow_is_f64 ? 2 : 1, n, nullptr, p, d_foe, nullptr, 0, nullptr, 0, d_phi, nullptr, nullptr,
                     h->d_stats_tmp, sizeof(mavd_frame_stats), 0, 0, (cudaStream_t)stream));
    if (d_max_phi) TRY(gather_max_phi_run(h->d_stats_tmp, n, d_max_phi, (cudaStream_t)stream));
    return MAVD_OK;
}

int mavd_debug_force_exact_residual(mavd_handle h, int32_t on) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "handle is NULL");
    DeviceGuard dg(h->cfg.device);
    MAVD_CUDA(cudaDeviceSynchronize());
    drop_graphs(h);
    h->force_exact_residual = on != 0;
    return MAVD_OK;
}

int mavd_residual_masks(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu,
                        const mavd_detect_params* prm, const double* d_foe, const uint8_t* d_sky, int64_t sky_stride,
                        const uint8_t* d_seg, int64_t seg_stride, void* d_phi, uint8_t* d_total, uint8_t* d_fixed,
                        mavd_frame_stats* d_stats, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "residual_masks"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_foe, MAVD_ERR_INVALID, "residual_masks: NULL buffer");
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    int n64 = 0, n32 = 0;
    TRY(upload_imu(h, h_imu, n, (cudaStream_t)stream, &n64, &n32));
    return residual_run(h, d_flow, 0, n, h->d_imu, p, d_foe, d_sky, sky_stride, d_seg, seg_stride, d_phi, d_total, d_fixed,
                        d_stats, sizeof(mavd_frame_stats), n64 > 0 ? (h->batch_rot > 0 ? 1 : 2) : 0, n32 > 0, (cudaStream_t)stream);
}

// A detection table request: max_det in range whenever there is a table.  The per-label workspace is allocated by the
// first request (outside any graph capture: every caller runs this before run_graphed).
static int check_det(mavd_handle h, int max_det, const void* det, const char* what) {
    if (!det) return MAVD_OK;
    MAVD_REQUIRE(max_det >= 1 && max_det <= MAVD_MAX_DETECTIONS, MAVD_ERR_INVALID, "%s: max_det %d outside 1..%d", what,
                 max_det, MAVD_MAX_DETECTIONS);
    MAVD_REQUIRE((reinterpret_cast<uintptr_t>(det) & 7) == 0, MAVD_ERR_INVALID, "%s: detections must be 8-byte aligned",
                 what);
    if (h->d_det_area) return MAVD_OK;
    TRY(h->arena.alloc(&h->d_det_area, (size_t)h->cfg.max_pairs * det_lab_stride(h)));
    return h->arena.alloc(&h->d_det_nlabels, (size_t)h->cfg.max_pairs);
}

int mavd_detections(mavd_handle h, const uint8_t* d_mask, int32_t n, const float* d_flow, const mavd_imu* h_imu,
                    int32_t max_det, mavd_detection* d_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "detections"));
    MAVD_REQUIRE(d_det != nullptr, MAVD_ERR_INVALID, "detections: NULL table");
    MAVD_REQUIRE(!d_flow || h_imu, MAVD_ERR_INVALID, "detections: a flow needs an imu array");
    TRY(check_det(h, max_det, d_det, "detections"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_mask != nullptr, MAVD_ERR_INVALID, "detections: NULL mask");
    const cudaStream_t s = (cudaStream_t)stream;
    if (d_flow) TRY(upload_imu(h, h_imu, n, s, nullptr, nullptr));
    const DetArgs da{d_det, max_det, h->d_det_area, det_lab_stride(h), d_flow, h->d_imu};
    return ccl_run(h, d_mask, n, nullptr, nullptr, 0, 0, h->d_det_nlabels, sizeof(int32_t), s, false, &da);
}

int mavd_good_features_to_track(mavd_handle h, const uint8_t* d_frames, int32_t n_frames, const mavd_gftt_params* prm,
                                const uint8_t* d_mask, int64_t mask_stride, float* d_corners, int32_t* d_count,
                                float* d_eig, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    MAVD_REQUIRE(h != nullptr && prm != nullptr, MAVD_ERR_INVALID, "good_features_to_track: NULL argument");
    const mavd_gftt_params p = *prm;
    MAVD_REQUIRE(n_frames >= 0 && n_frames <= h->max_frames, MAVD_ERR_INVALID,
                 "good_features_to_track: %d frames exceed the handle's %d", n_frames, h->max_frames);
    MAVD_REQUIRE(!std::isnan(p.quality_level) && !std::isnan(p.min_distance), MAVD_ERR_INVALID,
                 "good_features_to_track: NaN parameter");
    MAVD_REQUIRE(p.max_corners >= 0, MAVD_ERR_INVALID, "good_features_to_track: max_corners %d < 0", p.max_corners);
    MAVD_REQUIRE(mask_stride >= 0, MAVD_ERR_INVALID, "good_features_to_track: negative mask stride");
    MAVD_REQUIRE(p.block_size >= 1 && p.block_size <= 31, MAVD_ERR_UNSUPPORTED,
                 "good_features_to_track: block_size %d outside 1..31", p.block_size);
    MAVD_REQUIRE(p.gradient_size == 3, MAVD_ERR_UNSUPPORTED, "good_features_to_track: gradient_size must be 3");
    MAVD_REQUIRE(p.quality_level > 0, MAVD_ERR_UNSUPPORTED, "good_features_to_track: quality_level must be > 0");
    MAVD_REQUIRE(p.min_distance >= 0 && std::isfinite(p.min_distance), MAVD_ERR_UNSUPPORTED,
                 "good_features_to_track: min_distance must be finite and >= 0");
    MAVD_REQUIRE(std::isfinite(p.quality_level), MAVD_ERR_UNSUPPORTED, "good_features_to_track: infinite quality_level");
    if (n_frames == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && d_count && (d_corners || p.max_corners == 0), MAVD_ERR_INVALID,
                 "good_features_to_track: NULL buffer");
    return gftt_run(h, d_frames, n_frames, p, d_mask, d_mask ? mask_stride : 0, d_corners, d_count, d_eig,
                    (cudaStream_t)stream);
}

int mavd_pyr_lk(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_lk_params* prm,
                const float* d_prev_pts, int32_t n_points, const int32_t* d_n_points, float* d_next_pts,
                uint8_t* d_status, float* d_err, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    MAVD_REQUIRE(h != nullptr && prm != nullptr, MAVD_ERR_INVALID, "pyr_lk: NULL argument");
    const mavd_lk_params p = *prm;
    MAVD_REQUIRE(n_pairs >= 0 && n_pairs <= h->cfg.max_pairs, MAVD_ERR_INVALID, "pyr_lk: batch %d exceeds max_pairs %d",
                 n_pairs, h->cfg.max_pairs);
    MAVD_REQUIRE(pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    MAVD_REQUIRE(n_points >= 0 && n_points <= (1 << 24), MAVD_ERR_INVALID, "pyr_lk: n_points %d outside 0..2^24",
                 n_points);
    MAVD_REQUIRE(!std::isnan(p.criteria_eps) && !std::isnan(p.min_eig_threshold), MAVD_ERR_INVALID,
                 "pyr_lk: NaN parameter");
    MAVD_REQUIRE(p.win_w >= 3 && p.win_w <= 63 && p.win_h >= 3 && p.win_h <= 63, MAVD_ERR_UNSUPPORTED,
                 "pyr_lk: window %d x %d outside 3..63", p.win_w, p.win_h);
    MAVD_REQUIRE(p.max_level >= 0 && p.max_level <= MAVD_LK_MAX_LEVEL, MAVD_ERR_UNSUPPORTED,
                 "pyr_lk: max_level %d outside 0..%d", p.max_level, MAVD_LK_MAX_LEVEL);
    MAVD_REQUIRE(p.flags == 0 || p.flags == MAVD_LK_GET_MIN_EIGENVALS, MAVD_ERR_UNSUPPORTED,
                 "pyr_lk: flags %d not supported (0 or MAVD_LK_GET_MIN_EIGENVALS)", p.flags);
    MAVD_REQUIRE((p.criteria_type & ~(MAVD_TERM_COUNT | MAVD_TERM_EPS)) == 0, MAVD_ERR_UNSUPPORTED,
                 "pyr_lk: criteria_type %d not supported", p.criteria_type);
    if (n_pairs == 0 || n_points == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && d_prev_pts && d_next_pts && d_status && d_err, MAVD_ERR_INVALID, "pyr_lk: NULL buffer");
    return lk_run(h, d_frames, n_pairs, pair_stride, p, d_prev_pts, n_points, d_n_points, d_next_pts, d_status, d_err,
                  (cudaStream_t)stream);
}

int mavd_ccl(mavd_handle h, const uint8_t* d_mask, int32_t n, int32_t* d_labels, int32_t* d_boxes, int32_t max_boxes,
             int32_t* d_n_labels, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "ccl"));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_mask && d_n_labels, MAVD_ERR_INVALID, "ccl: NULL buffer");
    MAVD_REQUIRE(max_boxes >= 0, MAVD_ERR_INVALID, "ccl: max_boxes < 0");
    return ccl_run(h, d_mask, n, d_labels, max_boxes > 0 ? d_boxes : nullptr, (size_t)max_boxes * 5, max_boxes,
                   d_n_labels, sizeof(int32_t), (cudaStream_t)stream);
}

int mavd_magnitude(const void* d_flow, int32_t flow_is_f64, int64_t n_pixels, void* d_out, void* stream) {
    MAVD_REQUIRE(n_pixels >= 0 && (n_pixels == 0 || (d_flow && d_out)), MAVD_ERR_INVALID, "magnitude: bad arguments");
    if (n_pixels == 0) return MAVD_OK;
    return magnitude_run(d_flow, flow_is_f64 ? 1 : 0, n_pixels, d_out, (cudaStream_t)stream);
}

int mavd_simple_bbox(const uint8_t* d_img, int32_t width, int32_t height, int32_t channels, int32_t* d_out5,
                     void* stream) {
    MAVD_REQUIRE(d_img && d_out5 && width >= 1 && height >= 1 && channels >= 1, MAVD_ERR_INVALID,
                 "simple_bbox: bad arguments");
    return simple_bbox_run(d_img, width, height, channels, d_out5, (cudaStream_t)stream);
}

int mavd_tpr_fpr_counts(const uint8_t* d_gt, const int64_t* d_img, int64_t n, int64_t* d_counts4, void* stream) {
    MAVD_REQUIRE(n >= 0 && d_counts4 && (n == 0 || (d_gt && d_img)), MAVD_ERR_INVALID, "tpr_fpr_counts: bad arguments");
    return tpr_fpr_run(d_gt, d_img, n, d_counts4, (cudaStream_t)stream);
}

int mavd_phi_colormap(const void* d_phi, int32_t phi_is_f64, int64_t n_pixels, double max_value, uint8_t* d_gray_rgb,
                      uint8_t* d_bgr, void* stream) {
    MAVD_REQUIRE(n_pixels >= 0 && (n_pixels == 0 || d_phi) && (d_gray_rgb || d_bgr), MAVD_ERR_INVALID,
                 "phi_colormap: bad arguments");
    if (n_pixels == 0) return MAVD_OK;
    return phi_colormap_run(d_phi, phi_is_f64 ? 1 : 0, n_pixels, max_value, d_gray_rgb, d_bgr, (cudaStream_t)stream);
}

int mavd_mask_overlay(const uint8_t* d_frame, int32_t channels, const uint8_t* d_mask, int64_t n_pixels, uint8_t* d_out,
                      uint8_t* d_mask_rgb, void* stream) {
    MAVD_REQUIRE(n_pixels >= 0 && (channels == 1 || channels == 3) && (n_pixels == 0 || (d_frame && d_mask && d_out)),
                 MAVD_ERR_INVALID, "mask_overlay: bad arguments");
    if (n_pixels == 0) return MAVD_OK;
    return mask_overlay_run(d_frame, channels, d_mask, n_pixels, d_out, d_mask_rgb, (cudaStream_t)stream);
}

int mavd_flow_vis(const float* d_flow, int64_t n_pixels, uint8_t* d_bgr, uint32_t* d_scratch3, void* stream) {
    MAVD_REQUIRE(n_pixels >= 1 && d_flow && d_bgr && d_scratch3, MAVD_ERR_INVALID, "flow_vis: bad arguments");
    return flow_vis_run(d_flow, n_pixels, d_bgr, d_scratch3, (cudaStream_t)stream);
}

__global__ void records_fill_kernel(mavd_frame_record* rec, const double* foe, const int32_t* ninter, int n) {
    pdl_entry();
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    rec[f].foe[0] = foe[2 * f];
    rec[f].foe[1] = foe[2 * f + 1];
    rec[f].n_intersections = ninter[f];
}

static const mavd_aux_inputs kNoAux = {nullptr, 0, nullptr, 0, nullptr};

static int detect_run(mavd_handle h, const float* flow, int n, const mavd_detect_params& p, int n64, int n32,
                      const int32_t* d_samples, const mavd_aux_inputs& aux, uint8_t* d_total_out, uint8_t* fixed,
                      mavd_frame_record* d_records, int max_det, mavd_detection* d_det, cudaStream_t s) {
    char* stats0 = reinterpret_cast<char*>(d_records) + offsetof(mavd_frame_record, stats);
    // FoE estimation is one CTA per frame; what the residual kernel needs besides the FoE (zeroed statistics, the
    // segmentation maxima, an empty unit list) does not depend on it and runs on the side stream meanwhile
    const bool fork = h->s_aux != nullptr && !h->prof.on;
    if (fork) {
        MAVD_CUDA(cudaEventRecord(h->ev_fork, s));
        MAVD_CUDA(cudaStreamWaitEvent(h->s_aux, h->ev_fork, 0));
        pdl_break(h, 1);
        // the residual kernel lists the 128-pixel units of the fixed mask that hold foreground; the labelling passes
        // then visit only those (detection masks are almost empty)
        TRY(ccl_list_reset(h, n, h->s_aux, 1));
        TRY(residual_prepare(h, n, aux.seg, aux.seg_stride, reinterpret_cast<mavd_frame_stats*>(stats0),
                             sizeof(mavd_frame_record), h->s_aux, 1));
        MAVD_CUDA(cudaEventRecord(h->ev_join, h->s_aux));
    }
    TRY(foe_run(h, flow, 0, n, h->d_imu, p, d_samples, h->d_foe, h->d_ninter, s));
    if (fork) {
        MAVD_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
        pdl_break(h, 0);
    } else {
        TRY(ccl_list_reset(h, n, s));
    }
    TRY(residual_run(h, flow, 0, n, h->d_imu, p, h->d_foe, aux.sky, aux.sky_stride, aux.seg, aux.seg_stride, nullptr,
                     d_total_out, fixed, reinterpret_cast<mavd_frame_stats*>(stats0), sizeof(mavd_frame_record),
                     n64 > 0 ? (h->batch_rot > 0 ? 1 : 2) : 0, n32 > 0, s, true, aux.gt_flow, fork));
    int32_t* boxes0 = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(d_records) + offsetof(mavd_frame_record, boxes));
    char* nl0 = reinterpret_cast<char*>(d_records) + offsetof(mavd_frame_record, n_labels);
    const DetArgs da{d_det, max_det, h->d_det_area, det_lab_stride(h), flow, h->d_imu};
    TRY(ccl_run(h, fixed, n, nullptr, boxes0, sizeof(mavd_frame_record) / sizeof(int32_t), MAVD_MAX_BOXES,
                reinterpret_cast<int32_t*>(nl0), sizeof(mavd_frame_record), s, true, d_det ? &da : nullptr));
    MAVD_CUDA(launch_chained(pdl_next(h), records_fill_kernel, ceil_div(n, 128), 128, 0, s, d_records, h->d_foe, h->d_ninter, n));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Captured launch sequences.  One batch is ~50 launches on two streams; at small frame sizes (C1: one 640x480 pair)
// the launches, not the kernels, are the cost.  The sequence for a given argument tuple is captured once with stream
// capture (the side stream joins the capture through its fork / join events) and replayed as ONE graph launch.
// Everything that shapes the sequence is part of the key: buffers, batch geometry, detection parameters, which
// residual modes run.  The imu upload stays outside the graph (its contents change every call, the device buffer does
// not).  With profiling on, on a stream that is already being captured, or when capture fails, the launches go out
// directly — same kernels, same arguments.
// ------------------------------------------------------------------------------------------------
static constexpr size_t kMaxGraphs = 16;

struct KeyBuilder {
    std::vector<uint64_t> k;
    KeyBuilder& operator()(const void* p) { k.push_back((uint64_t)(uintptr_t)p); return *this; }
    KeyBuilder& operator()(int64_t v) { k.push_back((uint64_t)v); return *this; }
    KeyBuilder& operator()(const mavd_detect_params& p) {
        const size_t n = sizeof(p) / sizeof(uint64_t);
        uint64_t w[sizeof(mavd_detect_params) / sizeof(uint64_t)];
        memcpy(w, &p, sizeof(p));
        k.insert(k.end(), w, w + n);
        return *this;
    }
    KeyBuilder& operator()(const mavd_aux_inputs& a) {
        return (*this)(a.sky)(a.sky_stride)(a.seg)(a.seg_stride)((const void*)a.gt_flow);
    }
};

static void drop_graphs(mavd_handle h) {
    for (auto& g : h->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    h->graphs.clear();
}

template <typename F>
static int run_graphed(mavd_handle h, std::vector<uint64_t>&& key, cudaStream_t s, F&& body) {
    if (!h->tune.use_graph || h->prof.on || s == nullptr) return body(s);
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        return body(s);
    }
    for (auto& g : h->graphs) {
        if (g.key != key) continue;
        g.last_use = ++h->graph_clock;
        if (!g.exec) return body(s);        // this sequence could not be captured: direct launches
        MAVD_CUDA(cudaGraphLaunch(g.exec, s));
        g_launches.fetch_add(g.launches, std::memory_order_relaxed);
        return MAVD_OK;
    }
    mavd_handle_s::GraphEntry ent;
    ent.key = std::move(key);
    ent.last_use = ++h->graph_clock;
    const int64_t l0 = g_launches.load();
    int rc = MAVD_OK;
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
        rc = body(s);
        const cudaError_t e = cudaStreamEndCapture(s, &graph);
        const int64_t nl = g_launches.load() - l0;
        g_launches.fetch_sub(nl, std::memory_order_relaxed);        // captured, not run
        if (rc == MAVD_OK && e == cudaSuccess && graph &&
            cudaGraphInstantiate(&ent.exec, graph, 0) == cudaSuccess) {
            ent.launches = nl;
        } else {
            ent.exec = nullptr;
        }
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        if (rc != MAVD_OK) return rc;       // a real error (bad argument, failed launch configuration): report it
    } else {
        cudaGetLastError();
    }
    if (h->graphs.size() >= kMaxGraphs) {
        size_t lru = 0;
        for (size_t i = 1; i < h->graphs.size(); ++i)
            if (h->graphs[i].last_use < h->graphs[lru].last_use) lru = i;
        if (h->graphs[lru].exec) cudaGraphExecDestroy(h->graphs[lru].exec);
        h->graphs.erase(h->graphs.begin() + lru);
    }
    h->graphs.push_back(ent);
    if (!ent.exec) return body(s);
    MAVD_CUDA(cudaGraphLaunch(ent.exec, s));
    g_launches.fetch_add(ent.launches, std::memory_order_relaxed);
    return MAVD_OK;
}

// Work submitted on the legacy default stream (which cannot be captured) runs on the handle's own stream, ordered
// after / before the default stream by two events: same semantics for the caller.
struct StreamScope {
    mavd_handle h;
    cudaStream_t user, s;
    bool redirected = false;
    StreamScope(mavd_handle h_, void* stream) : h(h_), user((cudaStream_t)stream), s((cudaStream_t)stream) {
        if (user != nullptr || !h->tune.use_graph || h->prof.on || !h->s_main) return;
        if (cudaEventRecord(h->ev_main_in, user) != cudaSuccess ||
            cudaStreamWaitEvent(h->s_main, h->ev_main_in, 0) != cudaSuccess) {
            cudaGetLastError();
            return;
        }
        s = h->s_main;
        redirected = true;
    }
    ~StreamScope() {
        if (!redirected) return;
        if (cudaEventRecord(h->ev_main_out, s) != cudaSuccess || cudaStreamWaitEvent(user, h->ev_main_out, 0) != cudaSuccess)
            cudaGetLastError();
    }
};

extern "C" {

int mavd_farneback(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, float* d_flow,
                   void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n_pairs, "farneback"));
    MAVD_REQUIRE(pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    if (n_pairs == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && d_flow, MAVD_ERR_INVALID, "farneback: NULL buffer");
    StreamScope ss(h, stream);
    note_farneback_call(h, d_frames, n_pairs, pair_stride, d_flow);
    return run_graphed(h, std::move(KeyBuilder()(int64_t(1))(d_frames)(int64_t(n_pairs))(int64_t(pair_stride))(d_flow).k),
                       ss.s, [&](cudaStream_t s) { return farneback_run(h, d_frames, n_pairs, pair_stride, d_flow, s); });
}

int mavd_detect(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                const int32_t* d_samples, const mavd_aux_inputs* d_aux, uint8_t* d_total_out, uint8_t* d_fixed_out,
                mavd_frame_record* d_records, int32_t max_det, mavd_detection* d_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "detect"));
    TRY(check_det(h, max_det, d_det, "detect"));
    if (!d_det) max_det = 0;
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_flow && d_samples && d_records, MAVD_ERR_INVALID, "detect: NULL buffer");
    StreamScope ss(h, stream);
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    const mavd_aux_inputs aux = d_aux ? *d_aux : kNoAux;
    int n64 = 0, n32 = 0;
    TRY(upload_imu(h, h_imu, n, ss.s, &n64, &n32));
    uint8_t* fixed = d_fixed_out ? d_fixed_out : h->d_fixed;
    return run_graphed(h, std::move(KeyBuilder()(int64_t(2))(d_flow)(int64_t(n))(p)(int64_t(n64))(int64_t(h->batch_rot > 0))(int64_t(n32))(d_samples)(aux)
                                        (d_total_out)(fixed)(d_records)(int64_t(max_det))(d_det).k),
                       ss.s, [&](cudaStream_t s) {
                           return detect_run(h, d_flow, n, p, n64, n32, d_samples, aux, d_total_out, fixed, d_records,
                                             max_det, d_det, s);
                       });
}

// mavd_process (step false: pairs by pair_stride) and mavd_stream_process (step true: one new frame per id of h_ids)
static int process_run(mavd_handle h, const uint8_t* d_frames, int n_pairs, int pair_stride, bool step,
                       const int32_t* h_ids, const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* d_samples,
                       const mavd_aux_inputs* d_aux, float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out,
                       mavd_frame_record* d_records, int max_det, mavd_detection* d_det, void* stream) {
    const char* what = step ? "stream_process" : "process";
    MAVD_REQUIRE(!step || h_ids, MAVD_ERR_INVALID, "%s: ids array is NULL", what);
    TRY(check_batch(h, n_pairs, what));
    MAVD_REQUIRE(step || pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    TRY(check_det(h, max_det, d_det, what));
    if (!d_det) max_det = 0;
    if (n_pairs == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && d_samples && d_records, MAVD_ERR_INVALID, "%s: NULL buffer", what);
    if (step) TRY(check_stream_ids(h, h_ids, n_pairs, true, what));
    StreamScope ss(h, stream);
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    const mavd_aux_inputs aux = d_aux ? *d_aux : kNoAux;
    float* flow = d_flow_out ? d_flow_out : h->d_flow;
    uint8_t* fixed = d_fixed_out ? d_fixed_out : h->d_fixed;
    int n64 = 0, n32 = 0;
    TRY(upload_imu(h, h_imu, n_pairs, ss.s, &n64, &n32));
    if (step) TRY(upload_stream_slots(h, h_ids, n_pairs, ss.s));
    else note_farneback_call(h, d_frames, n_pairs, pair_stride, flow);
    const FrameSlots fs = h->stream_slots(n_pairs);
    TRY(run_graphed(h, std::move(KeyBuilder()(int64_t(step ? 5 : 3))(d_frames)(int64_t(n_pairs))(int64_t(pair_stride))(p)(int64_t(n64))(int64_t(h->batch_rot > 0))
                                        (int64_t(n32))(d_samples)(aux)(flow)(d_total_out)(fixed)(d_records)(int64_t(max_det))
                                        (d_det).k),
                    ss.s, [&](cudaStream_t s) {
                        TRY(farneback_run(h, d_frames, n_pairs, pair_stride, flow, s, step ? &fs : nullptr));
                        return detect_run(h, flow, n_pairs, p, n64, n32, d_samples, aux, d_total_out, fixed, d_records,
                                          max_det, d_det, s);
                    }));
    if (step) advance_streams(h, h_ids, n_pairs);
    return MAVD_OK;
}

int mavd_process(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                 const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                 float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                 int32_t max_det, mavd_detection* d_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return process_run(h, d_frames, n_pairs, pair_stride, false, nullptr, h_imu, prm, d_samples, d_aux, d_flow_out, d_total_out,
                       d_fixed_out, d_records, max_det, d_det, stream);
}

int mavd_stream_process(mavd_handle h, const uint8_t* d_frames, int32_t n, const int32_t* h_ids, const mavd_imu* h_imu,
                        const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                        float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                        int32_t max_det, mavd_detection* d_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return process_run(h, d_frames, n, 2, true, h_ids, h_imu, prm, d_samples, d_aux, d_flow_out, d_total_out, d_fixed_out,
                       d_records, max_det, d_det, stream);
}

// mavd_stream_farneback (step) and mavd_stream_start (expansions only)
static int stream_farneback_run(mavd_handle h, bool step, const uint8_t* d_frames, int n, const int32_t* h_ids,
                                float* d_flow, void* stream) {
    const char* what = step ? "stream_farneback" : "stream_start";
    MAVD_REQUIRE(h_ids != nullptr, MAVD_ERR_INVALID, "%s: ids array is NULL", what);
    TRY(check_batch(h, n, what));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && (d_flow || !step), MAVD_ERR_INVALID, "%s: NULL buffer", what);
    TRY(check_stream_ids(h, h_ids, n, step, what));
    StreamScope ss(h, stream);
    TRY(upload_stream_slots(h, h_ids, n, ss.s));
    const FrameSlots fs = h->stream_slots(n);
    const int n_pairs = step ? n : 0;
    TRY(run_graphed(h, std::move(KeyBuilder()(int64_t(step ? 4 : 6))(d_frames)(int64_t(n))(d_flow).k), ss.s,
                    [&](cudaStream_t s) { return farneback_run(h, d_frames, n_pairs, 2, d_flow, s, &fs); }));
    advance_streams(h, h_ids, n);
    return MAVD_OK;
}

int mavd_stream_start(mavd_handle h, const uint8_t* d_frames, int32_t n, const int32_t* h_ids, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return stream_farneback_run(h, false, d_frames, n, h_ids, nullptr, stream);
}

int mavd_stream_farneback(mavd_handle h, const uint8_t* d_frames, int32_t n, const int32_t* h_ids, float* d_flow,
                          void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return stream_farneback_run(h, true, d_frames, n, h_ids, d_flow, stream);
}

// ------------------------------------------------------------------------------------------------
// Host-buffer calls: three-stage pipeline over MAVD_HOST_SLOTS staging sets (copy-in stream, the caller's compute
// stream, copy-out stream).
// ------------------------------------------------------------------------------------------------
static int ensure_slot(mavd_handle h, int slot, bool want_flow_out, bool want_flow_in, bool want_bits_in, bool want_bits_out,
                       bool want_gt, bool want_det) {
    mavd_handle_s::HostSlot& S = h->slot[slot];
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
    const int B = h->cfg.max_pairs;
    Arena& A = h->arena;
    if (!S.d_frames) TRY(alloc_slot(h, S));
    if (want_flow_out && !S.d_flow) TRY(A.alloc(&S.d_flow, B * npx * 2));
    if (want_flow_in && !S.d_flow_in) TRY(A.alloc(&S.d_flow_in, B * npx * 2));
    if (want_bits_in && !S.d_bits_in) TRY(A.alloc(&S.d_bits_in, 2 * B * pb));
    if (want_bits_out && !S.d_bits_out) TRY(A.alloc(&S.d_bits_out, B * pb));
    if (want_gt && !S.d_gt_flow) TRY(A.alloc(&S.d_gt_flow, B * npx * 2));
    if (want_det && !S.d_det) TRY(A.alloc(&S.d_det, (size_t)B * MAVD_MAX_DETECTIONS));
    if (!h->s_in) MAVD_CUDA(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    if (!h->s_out) MAVD_CUDA(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    return MAVD_OK;
}

// np.random.randint(0, H, 2000) rows then np.random.randint(0, W, 2000) columns per frame (focus_of_expansion.py:69-71)
static int check_samples(const int32_t* h_samples, int n, int W, int Hh) {
    for (int f = 0; f < n; ++f) {
        const int32_t* sm = h_samples + (size_t)f * MAVD_SAMPLES_PER_FRAME;
        unsigned bad = 0;
        for (int i = 0; i < 2 * MAVD_N_SAMPLE_PAIRS; ++i) bad |= (unsigned)((unsigned)sm[i] >= (unsigned)Hh);
        for (int i = 2 * MAVD_N_SAMPLE_PAIRS; i < 4 * MAVD_N_SAMPLE_PAIRS; ++i) bad |= (unsigned)((unsigned)sm[i] >= (unsigned)W);
        MAVD_REQUIRE(!bad, MAVD_ERR_INVALID, "samples of frame %d out of range for a %dx%d frame (rows first, then columns)",
                     f, W, Hh);
    }
    return MAVD_OK;
}

// copy the optional per-frame host inputs of a batch into the slot's device buffers on the copy-in stream
static int stage_aux(mavd_handle h, mavd_handle_s::HostSlot& S, const mavd_aux_inputs& ha, int flags, int n,
                     cudaStream_t s_in, mavd_aux_inputs* da) {
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
    *da = kNoAux;
    if (ha.sky) {
        const int cnt = ha.sky_stride ? n : 1;
        if (flags & MAVD_HOST_SKY_PACKED) {
            uint8_t* bits = S.d_bits_in;
            MAVD_CUDA(cudaMemcpyAsync(bits, ha.sky, pb * cnt, cudaMemcpyHostToDevice, s_in));
            TRY(unpack_mask_run(bits, cnt, (int64_t)npx, 1, S.d_sky, s_in));
        } else {
            MAVD_CUDA(cudaMemcpyAsync(S.d_sky, ha.sky, npx * cnt, cudaMemcpyHostToDevice, s_in));
        }
        da->sky = S.d_sky;
        da->sky_stride = ha.sky_stride ? (int64_t)npx : 0;
    }
    if (ha.seg) {
        const int cnt = ha.seg_stride ? n : 1;
        if (flags & MAVD_HOST_SEG_PACKED) {
            uint8_t* bits = S.d_bits_in + (size_t)h->cfg.max_pairs * pb;
            MAVD_CUDA(cudaMemcpyAsync(bits, ha.seg, pb * cnt, cudaMemcpyHostToDevice, s_in));
            TRY(unpack_mask_run(bits, cnt, (int64_t)npx, 255, S.d_seg, s_in));
        } else {
            MAVD_CUDA(cudaMemcpyAsync(S.d_seg, ha.seg, npx * cnt, cudaMemcpyHostToDevice, s_in));
        }
        da->seg = S.d_seg;
        da->seg_stride = ha.seg_stride ? (int64_t)npx : 0;
    }
    if (ha.gt_flow) {
        MAVD_CUDA(cudaMemcpyAsync(S.d_gt_flow, ha.gt_flow, sizeof(float) * 2 * npx * n, cudaMemcpyHostToDevice, s_in));
        da->gt_flow = S.d_gt_flow;
    }
    return MAVD_OK;
}

static int check_aux_strides(mavd_handle h, const mavd_aux_inputs& a, int flags) {
    const int64_t npx = (int64_t)h->cfg.width * h->cfg.height, pb = packed_mask_bytes(npx);
    const int64_t sky_full = (flags & MAVD_HOST_SKY_PACKED) ? pb : npx, seg_full = (flags & MAVD_HOST_SEG_PACKED) ? pb : npx;
    MAVD_REQUIRE(a.sky_stride == 0 || a.sky_stride == sky_full, MAVD_ERR_INVALID, "sky_stride must be 0 or %lld",
                 (long long)sky_full);
    MAVD_REQUIRE(a.seg_stride == 0 || a.seg_stride == seg_full, MAVD_ERR_INVALID, "seg_stride must be 0 or %lld",
                 (long long)seg_full);
    return MAVD_OK;
}

// The arguments of a host-buffer call, all checked before anything is allocated or copied.  An empty batch reads no
// buffer.
static int check_host_args(mavd_handle h, const char* what, int n, const void* h_in, const int32_t* h_samples,
                           const mavd_frame_record* h_records, const mavd_aux_inputs& ha, int flags, int max_det,
                           const mavd_detection* h_det) {
    if (h_det)
        MAVD_REQUIRE(max_det >= 1 && max_det <= MAVD_MAX_DETECTIONS, MAVD_ERR_INVALID, "%s: max_det %d outside 1..%d",
                     what, max_det, MAVD_MAX_DETECTIONS);
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(h_in && h_samples && h_records, MAVD_ERR_INVALID, "%s: NULL buffer", what);
    TRY(check_aux_strides(h, ha, flags));
    return check_samples(h_samples, n, h->cfg.width, h->cfg.height);
}

// copy a batch's records, detection tables (when asked for) and estimate_fixed masks (packed first with
// MAVD_HOST_FIXED_PACKED) from the slot's device buffers to the caller's host buffers on stream s
static int copy_out(mavd_handle h, mavd_handle_s::HostSlot& S, int n, int flags, uint8_t* h_fixed_out,
                    mavd_frame_record* h_records, int max_det, mavd_detection* h_det, cudaStream_t s) {
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    MAVD_CUDA(cudaMemcpyAsync(h_records, S.d_records, sizeof(mavd_frame_record) * n, cudaMemcpyDeviceToHost, s));
    if (h_det)
        MAVD_CUDA(cudaMemcpyAsync(h_det, S.d_det, sizeof(mavd_detection) * max_det * n, cudaMemcpyDeviceToHost, s));
    if (h_fixed_out && (flags & MAVD_HOST_FIXED_PACKED)) {
        const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
        TRY(pack_mask_run(S.d_fixed, n, (int64_t)npx, S.d_bits_out, s));
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_bits_out, pb * n, cudaMemcpyDeviceToHost, s));
    } else if (h_fixed_out) {
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_fixed, npx * n, cudaMemcpyDeviceToHost, s));
    }
    return MAVD_OK;
}

// mavd_submit_host (step false: pairs by pair_stride) and mavd_stream_submit_host (step true: one new frame per id)
static int submit_host_run(mavd_handle h, int slot, const uint8_t* h_frames, int n_pairs, int pair_stride, bool step,
                           const int32_t* h_ids, const mavd_imu* h_imu, const mavd_detect_params* prm,
                           const int32_t* h_samples, const mavd_aux_inputs* h_aux, int flags, float* h_flow_out,
                           uint8_t* h_fixed_out, mavd_frame_record* h_records, int max_det, mavd_detection* h_det,
                           void* stream) {
    const char* what = step ? "stream_submit_host" : "submit_host";
    MAVD_REQUIRE(!step || h_ids, MAVD_ERR_INVALID, "%s: ids array is NULL", what);
    TRY(check_batch(h, n_pairs, what));
    MAVD_REQUIRE(slot >= 0 && slot < MAVD_HOST_SLOTS, MAVD_ERR_INVALID, "slot %d out of range", slot);
    MAVD_REQUIRE(step || pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    MAVD_REQUIRE(n_pairs >= 1, MAVD_ERR_INVALID, "%s: empty batch", what);
    const mavd_aux_inputs ha = h_aux ? *h_aux : kNoAux;
    TRY(check_host_args(h, what, n_pairs, h_frames, h_samples, h_records, ha, flags, max_det, h_det));
    if (step) TRY(check_stream_ids(h, h_ids, n_pairs, !(flags & MAVD_HOST_COPY_ONLY), what));
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const bool bgr = (flags & MAVD_HOST_BGR) != 0;
    TRY(ensure_slot(h, slot, h_flow_out != nullptr, false, (flags & (MAVD_HOST_SEG_PACKED | MAVD_HOST_SKY_PACKED)) != 0,
                    (flags & MAVD_HOST_FIXED_PACKED) && h_fixed_out, ha.gt_flow != nullptr, h_det != nullptr));
    mavd_handle_s::HostSlot& S = h->slot[slot];
    MAVD_REQUIRE(!S.busy, MAVD_ERR_INVALID, "slot %d is still in flight: call mavd_wait_host first", slot);
    const int n_frames = step ? n_pairs : pair_stride == 1 ? n_pairs + 1 : 2 * n_pairs;
    if (bgr && !S.d_bgr) TRY(h->arena.alloc(&S.d_bgr, (size_t)h->max_frames * npx * 3));
    StreamScope ss(h, stream);
    cudaStream_t s = ss.s;
    // copy-in stream (BGR frames are converted to gray there too, so the compute stream sees gray frames only)
    if (bgr) {
        MAVD_CUDA(cudaMemcpyAsync(S.d_bgr, h_frames, 3 * npx * n_frames, cudaMemcpyHostToDevice, h->s_in));
        TRY(bgr2gray_run(S.d_bgr, S.d_frames, (int64_t)npx * n_frames, h->s_in));
    } else {
        MAVD_CUDA(cudaMemcpyAsync(S.d_frames, h_frames, npx * n_frames, cudaMemcpyHostToDevice, h->s_in));
    }
    MAVD_CUDA(cudaMemcpyAsync(S.d_samples, h_samples, sizeof(int32_t) * MAVD_SAMPLES_PER_FRAME * n_pairs,
                              cudaMemcpyHostToDevice, h->s_in));
    mavd_aux_inputs da;
    TRY(stage_aux(h, S, ha, flags, n_pairs, h->s_in, &da));
    MAVD_CUDA(cudaEventRecord(S.ev_in, h->s_in));
    // compute stream (the caller's).  (Running the detection stages of a batch on a second stream, concurrently with
    // the next batch's Farneback, was measured: no gain, the GPU is already full and the work is only re-ordered.)
    MAVD_CUDA(cudaStreamWaitEvent(s, S.ev_in, 0));
    if (!(flags & MAVD_HOST_COPY_ONLY))
        TRY(process_run(h, S.d_frames, n_pairs, pair_stride, step, h_ids, h_imu, prm, S.d_samples, &da,
                        h_flow_out ? S.d_flow : nullptr, nullptr, S.d_fixed, S.d_records, max_det,
                        h_det ? S.d_det : nullptr, s));
    MAVD_CUDA(cudaEventRecord(S.ev_done, s));
    // copy-out stream
    MAVD_CUDA(cudaStreamWaitEvent(h->s_out, S.ev_done, 0));
    TRY(copy_out(h, S, n_pairs, flags, h_fixed_out, h_records, max_det, h_det, h->s_out));
    if (h_flow_out)
        MAVD_CUDA(cudaMemcpyAsync(h_flow_out, S.d_flow, sizeof(float) * 2 * npx * n_pairs, cudaMemcpyDeviceToHost, h->s_out));
    MAVD_CUDA(cudaEventRecord(S.ev_out, h->s_out));
    // the next batch's copy-in must not overwrite staging a kernel still reads: ordered by slot reuse rule
    S.busy = true;
    return MAVD_OK;
}

int mavd_submit_host(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                     const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                     const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                     mavd_frame_record* h_records, int32_t max_det, mavd_detection* h_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return submit_host_run(h, slot, h_frames, n_pairs, pair_stride, false, nullptr, h_imu, prm, h_samples, h_aux, flags,
                           h_flow_out, h_fixed_out, h_records, max_det, h_det, stream);
}

int mavd_stream_submit_host(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n, const int32_t* h_ids,
                            const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                            const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                            mavd_frame_record* h_records, int32_t max_det, mavd_detection* h_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    return submit_host_run(h, slot, h_frames, n, 2, true, h_ids, h_imu, prm, h_samples, h_aux, flags, h_flow_out, h_fixed_out,
                           h_records, max_det, h_det, stream);
}

int mavd_wait_host(mavd_handle h, int32_t slot) {
    MAVD_REQUIRE(h != nullptr, MAVD_ERR_INVALID, "wait_host: handle is NULL");
    MAVD_REQUIRE(slot >= 0 && slot < MAVD_HOST_SLOTS, MAVD_ERR_INVALID, "slot %d out of range", slot);
    mavd_handle_s::HostSlot& S = h->slot[slot];
    if (!S.busy) return MAVD_OK;
    DeviceGuard dg(h->cfg.device);
    S.busy = false;
    MAVD_CUDA(cudaEventSynchronize(S.ev_out));
    return MAVD_OK;
}

int mavd_detect_host(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                     const mavd_detect_params* prm, const int32_t* h_samples, const mavd_aux_inputs* h_aux,
                     int32_t flags, uint8_t* h_fixed_out, mavd_frame_record* h_records, int32_t max_det,
                     mavd_detection* h_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "detect_host"));
    const mavd_aux_inputs ha = h_aux ? *h_aux : kNoAux;
    TRY(check_host_args(h, "detect_host", n, h_flow, h_samples, h_records, ha, flags, max_det, h_det));
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE((flags & MAVD_HOST_BGR) == 0, MAVD_ERR_INVALID, "detect_host: MAVD_HOST_BGR has no meaning here");
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    TRY(mavd_wait_host(h, 0));
    TRY(ensure_slot(h, 0, false, true, (flags & (MAVD_HOST_SEG_PACKED | MAVD_HOST_SKY_PACKED)) != 0,
                    (flags & MAVD_HOST_FIXED_PACKED) && h_fixed_out, ha.gt_flow != nullptr, h_det != nullptr));
    mavd_handle_s::HostSlot& S = h->slot[0];
    StreamScope ss(h, stream);
    cudaStream_t s = ss.s;
    MAVD_CUDA(cudaMemcpyAsync(S.d_flow_in, h_flow, sizeof(float) * 2 * npx * n, cudaMemcpyHostToDevice, s));
    MAVD_CUDA(cudaMemcpyAsync(S.d_samples, h_samples, sizeof(int32_t) * MAVD_SAMPLES_PER_FRAME * n, cudaMemcpyHostToDevice, s));
    mavd_aux_inputs da;
    TRY(stage_aux(h, S, ha, flags, n, s, &da));
    if (!(flags & MAVD_HOST_COPY_ONLY))
        TRY(mavd_detect(h, S.d_flow_in, n, h_imu, prm, S.d_samples, &da, nullptr, S.d_fixed, S.d_records, max_det,
                        h_det ? S.d_det : nullptr, s));
    TRY(copy_out(h, S, n, flags, h_fixed_out, h_records, max_det, h_det, s));
    MAVD_CUDA(cudaStreamSynchronize(s));
    return MAVD_OK;
}

int64_t mavd_packed_mask_bytes(int32_t width, int32_t height) {
    if (width <= 0 || height <= 0) return 0;
    return packed_mask_bytes((int64_t)width * height);
}

int mavd_pack_mask(const uint8_t* d_mask, int32_t n, int64_t n_pixels, uint8_t* d_bits, void* stream) {
    MAVD_REQUIRE(n >= 0 && n <= 65535 && n_pixels >= 1 && (n == 0 || (d_mask && d_bits)), MAVD_ERR_INVALID,
                 "pack_mask: bad arguments");
    MAVD_REQUIRE((reinterpret_cast<uintptr_t>(d_bits) & 3) == 0, MAVD_ERR_INVALID, "pack_mask: d_bits must be 4-byte aligned");
    if (n == 0) return MAVD_OK;
    return pack_mask_run(d_mask, n, n_pixels, d_bits, (cudaStream_t)stream);
}

int mavd_unpack_mask(const uint8_t* d_bits, int32_t n, int64_t n_pixels, uint8_t value, uint8_t* d_mask, void* stream) {
    MAVD_REQUIRE(n >= 0 && n <= 65535 && n_pixels >= 1 && (n == 0 || (d_mask && d_bits)), MAVD_ERR_INVALID,
                 "unpack_mask: bad arguments");
    MAVD_REQUIRE((reinterpret_cast<uintptr_t>(d_bits) & 3) == 0, MAVD_ERR_INVALID, "unpack_mask: d_bits must be 4-byte aligned");
    if (n == 0) return MAVD_OK;
    return unpack_mask_run(d_bits, n, n_pixels, value, d_mask, (cudaStream_t)stream);
}

}  // extern "C"
