// Shared helpers for libmavd (sm_100a).  Error reporting never throws across the C ABI.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <vector>

#include "mavd.h"

namespace mavd {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

#define MAVD_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            ::mavd::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
            return (e__ == cudaErrorMemoryAllocation) ? MAVD_ERR_NOMEM : MAVD_ERR_CUDA;          \
        }                                                                                       \
    } while (0)

// Call after every kernel launch: counts the launch and surfaces configuration errors.
#define MAVD_LAUNCHED()                                                                         \
    do {                                                                                        \
        ::mavd::g_launches.fetch_add(1, std::memory_order_relaxed);                             \
        MAVD_CUDA(cudaGetLastError());                                                          \
    } while (0)

#define TRY_RC(...)                                                                             \
    do {                                                                                        \
        int rc__ = (__VA_ARGS__);                                                                       \
        if (rc__ != MAVD_OK) return rc__;                                                       \
    } while (0)

#define MAVD_REQUIRE(cond, code, ...)                                                           \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            ::mavd::set_error(__VA_ARGS__);                                                     \
            return (code);                                                                      \
        }                                                                                       \
    } while (0)

// Switches to a handle's device for the lifetime of the guard and restores the caller's current device afterwards
// (every handle-taking entry point of the C ABI holds one).
struct DeviceGuard {
    int prev = -1, cur = -1;
    explicit DeviceGuard(int dev) {
        if (dev < 0) return;
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
        cur = dev;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != cur) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: opt in once per (kernel, device).
template <auto Kernel>
static inline cudaError_t ensure_dynamic_smem(size_t bytes) {
    static std::atomic<uint64_t> done{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = dev < 64 ? (1ull << dev) : 0ull;
    if (bit && (done.load(std::memory_order_acquire) & bit)) return cudaSuccess;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess && bit) done.fetch_or(bit, std::memory_order_release);
    return e;
}

// ------------------------------------------------------------------------------------------------
// Programmatic dependent launch.  One batch is ~50 kernels, each consuming what its predecessor on the stream wrote.
// A kernel launched through launch_chained(pdl = true) is set up while the predecessor's last CTAs drain (a CTA that
// exits counts as having released its dependents) instead of after the whole grid has retired; pdl_entry(), the FIRST
// statement of every such kernel (before any early exit and before any global access), holds its CTAs until the
// predecessor grid has completed and its writes are visible.  What leaves the critical path is the launch itself:
// block scheduling, parameter / descriptor fetch, the ramp of the first wave (C1, one 640x480 pair: 0.255 -> 0.245 ms
// per pair; C2: +0.4..1.4 %).  Without the launch attribute the instruction does nothing.
// Every CTA of a chained kernel must execute pdl_entry(): a grid whose CTAs all left without waiting would complete
// before its predecessor and release its successor too early.
// (Releasing the dependents explicitly at kernel entry, griddepcontrol.launch_dependents, was measured and dropped:
// the successor's CTAs then sit in the slots the predecessor's tail frees and the side stream's kernels wait for
// them: C2 -2 %, C1 -10 %.)
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_entry() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_chained(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                         cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

constexpr int kMaxPolyN = 8;
constexpr int kMaxLevels = 16;
constexpr int kMaxWinHalf = 31;

// One pyramid level: geometry, resize/blur tables and per-level buffers (all device memory).
struct Level {
    int k = 0;
    double scale = 1.0;
    int w = 0, h = 0;
    int pitch = 0;      // floats per row, multiple of 64 so 64-wide tiles never leave the row
    size_t plane = 0;   // pitch * h
    int ksz = 3;
    float sigma = 0.f;
    // pyramid tables (full-res -> this level): combined blur+resize filter of ksz+1 taps per output sample
    int* xbase = nullptr;  float* xtab = nullptr;   // [w], [w][ksz+1]
    float* xtabT = nullptr;                         // [taps][w]: xtab tap-major (staged horizontal pyramid pass)
    int hspan_max = 0;                              // largest source span of 64 adjacent outputs (+ taps)
    int hstride_min = 0;                            // smallest distance between the sources of adjacent outputs
    int* ybase = nullptr;  float* ytab = nullptr;   // [h], [h][ksz+1]
    float* tmp = nullptr;                           // [frames][h][Wp] vertical pass output (levels >= 1)
    // exact power-of-two level (farneback.cu: HalfPyr): every output sample has the same ksz + 1 weights and its window
    // starts 2^k samples after its neighbour's; host copies of those weights for the kernels that exploit it
    bool x_half = false, y_half = false;
    float xwt[160] = {}, ywt[160] = {};
    // flow upsample tables (next-coarser level -> this level)
    int* fxi0 = nullptr; float* fxa = nullptr;  // [w]
    int* fyi0 = nullptr; float* fya = nullptr;  // [h]
    // buffers
    float* img = nullptr;   // [frames][h][pitch]
    float* R = nullptr;     // [frames][5][h][pitch]
    float* M[2] = {nullptr, nullptr};  // [pairs][5][h][pitch]
    float* flow = nullptr;  // [pairs][h][pitch] float2 (unused for level 0: written to the caller's buffer)
    int last_m = 0;         // which M buffer holds the last update (for taps)
    CUtensorMap tmapM[2];   // TMA descriptors of M[0] / M[1]: dims {pitch, h, pairs*5}, box {80, 32+2m, 5}
    CUtensorMap tmapR;      // TMA descriptor of R: dims {pitch, h, frames*5}, box {80, 48, 10} (L2 prefetch only)
    CUtensorMap tmapRbox;   // TMA descriptor of R with the M box geometry {80, 32+2m, 5}: R1 staged in shared memory
    bool has_tmap = false;
    CUtensorMap tmapM16[2]; // the same with 64 x 16 tiles: box {80, 16+2m, 5}
    CUtensorMap tmapRbox16;
    bool has_tmap16 = false;
    CUtensorMap tmapImg;    // TMA descriptor of img: dims {pitch, h, frames}, box {80, 32+2 poly_n, 1} (polynomial expansion)
    bool has_tmap_img = false;
};

// Optional per-kernel-class timing with CUDA events on the launching stream (bench.py's roofline).
struct Profiler {
    struct Rec { int cls; cudaEvent_t a, b; };
    bool on = false;
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        return e;
    }
};

struct ProfScope {
    Profiler* p;
    cudaStream_t s;
    size_t idx = 0;
    ProfScope(Profiler* prof, int cls, cudaStream_t st) : p(prof && prof->on ? prof : nullptr), s(st) {
        if (!p) return;
        Profiler::Rec r{cls, p->get(), p->get()};
        cudaEventRecord(r.a, s);
        idx = p->recs.size();
        p->recs.push_back(r);
    }
    ~ProfScope() {
        if (p) cudaEventRecord(p->recs[idx].b, s);
    }
};

struct PolyConst {
    float g[kMaxPolyN + 1], xg[kMaxPolyN + 1], xxg[kMaxPolyN + 1];
    float ig11, ig03, ig33, ig55;
    int n;
};

}  // namespace mavd

struct mavd_handle_s {
    mavd_config cfg;
    int n_levels = 0;               // number of pyramid images
    mavd::Level lv[mavd::kMaxLevels];  // lv[0] = finest (k = 0)
    mavd::PolyConst poly;
    float* gauss_win = nullptr;     // [m+1] device, FarnebackUpdateFlow_GaussianBlur half kernel
    int max_frames = 0;
    size_t bytes = 0;
    // detection workspace
    mavd_imu* d_imu = nullptr;      // [max_pairs]
    double* d_foe = nullptr;        // [max_pairs][2]
    int32_t* d_ninter = nullptr;    // [max_pairs]
    int32_t* d_labels = nullptr;    // [max_pairs][H][W]
    int32_t* d_scan = nullptr;      // CCL scratch
    double* d_xn = nullptr;         // [W] -(x/w - 0.5)*2, detector.py:90 (host-built, IEEE identical to NumPy)
    double* d_yn = nullptr;         // [H] -(y/h - 0.5)*2, detector.py:91
    mavd_frame_stats* d_stats_tmp = nullptr;  // [max_pairs] scratch for mavd_get_phi
    bool force_exact_residual = false;        // tests: disable the float32 pre-decision
    uint8_t* d_total = nullptr;     // [max_pairs][H][W]
    uint8_t* d_fixed = nullptr;
    float* d_flow = nullptr;        // [max_pairs][H][W][2] (when the caller does not want the flow)
    // detection tables (allocated by the first call that asks for one: mavd_workspace_bytes is unchanged otherwise)
    int32_t* d_det_area = nullptr;  // [max_pairs][det_lab_stride]: area per label, then -(slot + 1) of a selected label
    int32_t* d_det_nlabels = nullptr;   // [max_pairs] label counts of mavd_detections
    // sparse features (allocated by the first call that needs them: mavd_workspace_bytes is unchanged otherwise)
    void* sp_gftt = nullptr;        // corner workspace of mavd::gftt_chunk() frames (sparse.cu: gftt_run)
    uint8_t* sp_pyr = nullptr;      // [max_frames] pyramid levels 1.. of mavd_pyr_lk
    short2* sp_der = nullptr;       // [max_frames] int16 Scharr derivatives of every level
    // host-path staging: MAVD_HOST_SLOTS independent sets of device buffers + the streams/events that let
    // the H2D of one batch, the compute of the previous one and the D2H of the one before overlap
    struct HostSlot {
        uint8_t* d_frames = nullptr;    // [max_frames][H][W]
        uint8_t* d_bgr = nullptr;       // [max_frames][H][W][3], mavd_submit_host_bgr only (allocated on first use)
        int32_t* d_samples = nullptr;   // [max_pairs][4000]
        uint8_t* d_sky = nullptr;       // [max_pairs][H][W]
        uint8_t* d_seg = nullptr;
        float* d_flow_in = nullptr;     // [max_pairs][H][W][2], mavd_detect_host only (allocated on first use)
        mavd_frame_record* d_records = nullptr;
        uint8_t* d_fixed = nullptr;     // [max_pairs][H][W] estimate_fixed masks of the batch
        uint8_t* d_bits_in = nullptr;   // [2][max_pairs][packed bytes]: segmentation / sky as they cross the bus at
                                        // 1 bit per pixel (allocated on first use)
        uint8_t* d_bits_out = nullptr;  // [max_pairs][packed bytes]: estimate_fixed packed for the way back
        float* d_gt_flow = nullptr;     // [max_pairs][H][W][2] ground-truth flow (allocated on first use)
        float* d_flow = nullptr;        // [max_pairs][H][W][2] flow of the batch (allocated on first request)
        mavd_detection* d_det = nullptr;    // [max_pairs][MAVD_MAX_DETECTIONS] detection tables (allocated on first request)
        cudaEvent_t ev_in = nullptr, ev_done = nullptr, ev_out = nullptr;
        bool busy = false;
    } slot[MAVD_HOST_SLOTS];
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaStream_t s_aux = nullptr;     // high-priority side stream for the coarse pyramid levels (farneback_run)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_pyr = nullptr;
    mavd_tuning tune;                 // launch-shape choices (mavd_set_tuning); results never depend on them
    mavd::Profiler prof;
    // imu staging: callers' imu arrays are copied into a ring of pinned slots before the asynchronous upload, so the
    // call never retains the caller's pointer; an event per slot keeps a slot from being rewritten while its copy
    // is still pending
    static constexpr int kImuRing = 8;
    mavd_imu* h_imu_ring = nullptr;   // pinned, [kImuRing][max_pairs]
    cudaEvent_t imu_ev[kImuRing] = {};
    int imu_next = 0;
    // captured launch sequences (api.cu: run_graphed), least recently used entry replaced first
    struct GraphEntry {
        std::vector<uint64_t> key;
        cudaGraphExec_t exec = nullptr;
        int64_t launches = 0;
        uint64_t last_use = 0;
    };
    std::vector<GraphEntry> graphs;
    uint64_t graph_clock = 0;
    cudaStream_t s_main = nullptr;    // work submitted on the legacy default stream runs here between two events
    cudaEvent_t ev_main_in = nullptr, ev_main_out = nullptr;
    bool force_generic_iter = false;  // tests: run the non-TMA iteration kernel
    int batch_rot = 0;                // frames of the last uploaded imu array that derotate by a non-zero rotation
    // programmatic dependent launch (pdl_next / pdl_break below): may the next kernel on the caller's stream [0] /
    // the side stream [1] be chained to the kernel launched before it on that stream?
    bool pdl_ok[2] = {false, false};
    // last call bookkeeping for taps
    int last_pairs = 0, last_stride = 1;
    float* last_flow0 = nullptr;
    const uint8_t* last_frames = nullptr;
};

namespace mavd {
// Launch attribute of the next kernel on lane 0 (the caller's stream) or 1 (the side stream): chained when the previous
// operation on that stream was one of this library's chained kernels.  pdl_break() after anything else (event waits,
// memsets, copies, the start of a call), so that a programmatic edge only ever joins two kernels that both execute
// pdl_entry().  Off under the per-class profiler, whose event records sit between the kernels.
static inline bool pdl_next(mavd_handle h, int lane = 0) {
    const bool chained = h->tune.use_pdl != 0 && !h->prof.on && h->pdl_ok[lane];
    h->pdl_ok[lane] = true;
    return chained;
}
static inline void pdl_break(mavd_handle h, int lane = 0) { h->pdl_ok[lane] = false; }

// api.cu
bool encode_tensor_map_3d(CUtensorMap* map, bool is_u8, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                          uint64_t s1_bytes, uint64_t s2_bytes, uint32_t b0, uint32_t b1, uint32_t b2);
// farneback.cu
int farneback_run(mavd_handle h, const uint8_t* d_frames, int n_pairs, int pair_stride, float* d_flow,
                  cudaStream_t s);
int farneback_tap(mavd_handle h, int kind, int level, int index, float* d_out, cudaStream_t s);
// detect.cu
int bgr2gray_run(const uint8_t* d_bgr, uint8_t* d_gray, int64_t n, cudaStream_t s);
int derotate_run(mavd_handle h, const void* d_flow, int flow_is_f64, int n, const mavd_imu* d_imu, double* d_out,
                 cudaStream_t s);
int foe_run(mavd_handle h, const void* d_flow, int flow_kind, int n, const mavd_imu* d_imu,
            const mavd_detect_params& prm, const int32_t* d_samples, double* d_foe, int32_t* d_ninter, cudaStream_t s);
int ransac_run(const double* d_estimates, int K, double threshold, double* d_out, cudaStream_t s);
int gather_max_phi_run(const mavd_frame_stats* d_stats, int n, double* d_out, cudaStream_t s);
int residual_run(mavd_handle h, const void* d_flow, int flow_kind, int n, const mavd_imu* d_imu, const mavd_detect_params& prm,
                 const double* d_foe, const uint8_t* d_sky, int64_t sky_stride, const uint8_t* d_seg,
                 int64_t seg_stride, void* d_phi, uint8_t* d_total, uint8_t* d_fixed, mavd_frame_stats* d_stats,
                 size_t stats_stride_bytes, int run_f64, int run_f32, cudaStream_t s, bool list_fixed_units = false,
                 const float* d_gt_flow = nullptr, bool prepared = false);
// the part of residual_run that does not depend on the flow or the FoE (lane: common.cuh pdl_next); a caller that ran
// it passes prepared = true
int residual_prepare(mavd_handle h, int n, const uint8_t* d_seg, int64_t seg_stride, mavd_frame_stats* d_stats,
                     size_t stats_stride_bytes, cudaStream_t s, int lane);
int phi_colormap_run(const void* d_phi, int is_f64, int64_t n, double max_value, uint8_t* d_gray_rgb, uint8_t* d_bgr,
                     cudaStream_t s);
int mask_overlay_run(const uint8_t* d_frame, int channels, const uint8_t* d_mask, int64_t n, uint8_t* d_out,
                     uint8_t* d_mask_rgb, cudaStream_t s);
int pack_mask_run(const uint8_t* d_mask, int n, int64_t npx, uint8_t* d_bits, cudaStream_t s);
int unpack_mask_run(const uint8_t* d_bits, int n, int64_t npx, uint8_t value, uint8_t* d_mask, cudaStream_t s);
static inline int64_t packed_mask_bytes(int64_t npx) { return ((npx + 7) / 8 + 3) / 4 * 4; }
// The labelling passes walk a list of occupied 128-pixel units of the mask.  residual_run(list_fixed_units) appends the
// units of the fixed mask while it writes it (after ccl_list_reset), so that ccl_run(list_ready) never streams the mask.
int ccl_list_reset(mavd_handle h, int n, cudaStream_t s, int lane = 0);
int ccl_n_units(mavd_handle h);
int* ccl_unit_marks(mavd_handle h);
int* ccl_unit_list(mavd_handle h);
int* ccl_unit_count(mavd_handle h);
int magnitude_run(const void* d_flow, int is_f64, int64_t n, void* d_out, cudaStream_t s);
int simple_bbox_run(const uint8_t* d_img, int w, int h, int c, int32_t* d_out5, cudaStream_t s);
int tpr_fpr_run(const uint8_t* d_gt, const int64_t* d_img, int64_t n, int64_t* d_counts4, cudaStream_t s);
int flow_vis_run(const float* d_flow, int64_t n, uint8_t* d_bgr, uint32_t* d_scratch3, cudaStream_t s);
// Detection table of ccl_run: the max_det largest components of each frame (include/mavd.h: mavd_detection).
struct DetArgs {
    mavd_detection* det;     // [n][max_det]
    int max_det;
    int32_t* lab_area;       // h->d_det_area
    int lab_stride;          // det_lab_stride(h)
    const float* flow;       // nullable: (n, H, W, 2) float32, derotated per pixel as mavd_derotate does
    const mavd_imu* imu;     // device, n entries (with flow)
};
// labels a frame can hold under 8-connectivity (one per 2 x 2 block at most), plus the unused label 0
static inline int det_lab_stride(mavd_handle h) { return ((h->cfg.width + 1) / 2) * ((h->cfg.height + 1) / 2) + 1; }
int ccl_run(mavd_handle h, const uint8_t* d_mask, int n, int32_t* d_labels, int32_t* d_boxes, size_t boxes_stride,
            int max_boxes, int32_t* d_n_labels, size_t nlabels_stride_bytes, cudaStream_t s, bool list_ready = false,
            const DetArgs* det = nullptr);
// sparse.cu: corners and pyramidal Lucas-Kanade
struct GfttWork {
    float3* cov;                    // [chunk][H][W] products of the Sobel derivatives
    double* rows;                   // [chunk][H][W][3] row sums of the block
    float* eig;                     // [chunk][H][W] when the caller wants no eig image
    unsigned long long* keys;       // [chunk][gftt_key_cap] candidates
    int* grid;                      // [chunk][gftt_grid_cap] accepted corners by cell
    uint32_t* maxv;                 // [chunk]
    int* n_cand;                    // [chunk]
};
size_t gftt_key_cap(int W, int H);
size_t gftt_grid_cap(int W, int H);
int gftt_chunk();
int gftt_run(mavd_handle h, const GfttWork& ws, const uint8_t* d_frames, int n, const mavd_gftt_params& p,
             const uint8_t* d_mask, int64_t mask_stride, float* d_corners, int32_t* d_count, float* d_eig,
             cudaStream_t s);
size_t lk_pyr_frame_bytes(int W, int H);
size_t lk_der_frame_elems(int W, int H);
int lk_run(mavd_handle h, uint8_t* pyr, short2* der, const uint8_t* d_frames, int n_pairs, int pair_stride,
           const mavd_lk_params& p, const float* d_prev, int n_points, const int32_t* d_n_points, float* d_next,
           uint8_t* d_status, float* d_err, cudaStream_t s);
}  // namespace mavd
