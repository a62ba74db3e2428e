// C ABI of libmavd (include/mavd.h): handle lifecycle, parameter tables, stage entry points and the
// whole-path calls.  No exceptions cross this boundary; every failure is an int status plus a
// thread-local message.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
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

static inline int cv_round(double v) { return (int)nearbyint(v); }  // round-half-even, like cvRound

// cv::resize(INTER_LINEAR) source index / weight per destination index (pixel-centre mapping).
static void resize_tables(int src, int dst, std::vector<int>& i0, std::vector<float>& a) {
    i0.resize(dst);
    a.resize(dst);
    const double inv_scale = (double)dst / src;
    const double scale = 1.0 / inv_scale;
    for (int d = 0; d < dst; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s = (int)floorf(f);
        float w = f - (float)s;
        if (s < 0) { s = 0; w = 0.f; }
        if (s >= src - 1) { s = src - 1; w = 0.f; }
        i0[d] = s;
        a[d] = w;
    }
}

// cv::getGaussianKernel(ksz, sigma, CV_32F)
static std::vector<float> gaussian_kernel(int ksz, double sigma) {
    std::vector<float> k(ksz);
    if (sigma <= 0 && ksz == 3) { k[0] = 0.25f; k[1] = 0.5f; k[2] = 0.25f; return k; }
    if (sigma <= 0) sigma = ((ksz - 1) * 0.5 - 1) * 0.3 + 0.8;
    std::vector<double> t(ksz);
    double sum = 0;
    for (int i = 0; i < ksz; ++i) {
        double x = i - (ksz - 1) * 0.5;
        t[i] = exp(-0.5 * x * x / (sigma * sigma));
        sum += t[i];
    }
    for (int i = 0; i < ksz; ++i) k[i] = (float)(t[i] / sum);
    return k;
}

// FarnebackPrepareGaussian: taps and the four needed entries of inv(G) (Appendix A of SURVEY.md).
static int poly_setup(int n, double sigma, PolyConst& pc) {
    if (sigma < 1.1920929e-07) sigma = n * 0.3;
    float g[2 * kMaxPolyN + 1], xg[2 * kMaxPolyN + 1], xxg[2 * kMaxPolyN + 1];
    double s = 0;
    for (int x = -n; x <= n; ++x) {
        g[x + n] = (float)exp(-x * x / (2 * sigma * sigma));
        s += g[x + n];
    }
    s = 1. / s;
    for (int x = -n; x <= n; ++x) {
        g[x + n] = (float)(g[x + n] * s);
        xg[x + n] = (float)(x * g[x + n]);
        xxg[x + n] = (float)(x * x * g[x + n]);
    }
    double G[6][6];
    memset(G, 0, sizeof(G));
    for (int y = -n; y <= n; ++y)
        for (int x = -n; x <= n; ++x) {
            const float gg = g[y + n] * g[x + n];
            G[0][0] += gg;
            G[1][1] += gg * x * x;
            G[3][3] += gg * x * x * x * x;
            G[5][5] += gg * x * x * y * y;
        }
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    // Gauss-Jordan inverse of the 6x6 (symmetric positive definite) matrix
    double A[6][12];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 12; ++j) A[i][j] = j < 6 ? G[i][j] : (j - 6 == i ? 1.0 : 0.0);
    for (int c = 0; c < 6; ++c) {
        int piv = c;
        for (int r = c + 1; r < 6; ++r)
            if (fabs(A[r][c]) > fabs(A[piv][c])) piv = r;
        if (fabs(A[piv][c]) < 1e-300) return MAVD_ERR_INVALID;
        if (piv != c)
            for (int j = 0; j < 12; ++j) { double t = A[c][j]; A[c][j] = A[piv][j]; A[piv][j] = t; }
        const double d = A[c][c];
        for (int j = 0; j < 12; ++j) A[c][j] /= d;
        for (int r = 0; r < 6; ++r)
            if (r != c) {
                const double f = A[r][c];
                if (f != 0)
                    for (int j = 0; j < 12; ++j) A[r][j] -= f * A[c][j];
            }
    }
    pc.n = n;
    for (int k = 0; k <= kMaxPolyN; ++k) {
        pc.g[k] = k <= n ? g[n + k] : 0.f;
        pc.xg[k] = k <= n ? xg[n + k] : 0.f;
        pc.xxg[k] = k <= n ? xxg[n + k] : 0.f;
    }
    pc.ig11 = (float)A[1][6 + 1];
    pc.ig03 = (float)A[0][6 + 3];
    pc.ig33 = (float)A[3][6 + 3];
    pc.ig55 = (float)A[5][6 + 5];
    return MAVD_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// TMA descriptor of a rank-3 tensor {d0, d1, d2} (d0 fastest) of 4-byte floats or bytes with byte strides s1, s2 and a
// box {b0, b1, b2}; out-of-bounds cells are filled with zeros.  Base and strides must be multiples of 16 bytes.
bool encode_tensor_map_3d(CUtensorMap* map, bool is_u8, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                          uint64_t s1_bytes, uint64_t s2_bytes, uint32_t b0, uint32_t b1, uint32_t b2) {
    static std::atomic<EncodeTiledFn> fn_cache{nullptr};
    EncodeTiledFn fn = fn_cache.load();
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || !f) {
            cudaGetLastError();
            return false;
        }
        fn = (EncodeTiledFn)f;
        fn_cache.store(fn);
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (s1_bytes & 15) || (s2_bytes & 15)) return false;
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {s1_bytes, s2_bytes};
    cuuint32_t box[3] = {b0, b1, b2};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = fn(map, is_u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                    const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// TMA descriptor of a planar buffer: rank-3 float tensor {pitch, h, planes}, box {80, box_h, box_planes}, zero fill.
static bool make_plane_tensor_map(CUtensorMap* map, float* base, int pitch, int h, int planes, size_t plane, int box_h,
                                  int box_planes) {
    return encode_tensor_map_3d(map, false, base, (uint64_t)pitch, (uint64_t)h, (uint64_t)planes,
                                (uint64_t)pitch * sizeof(float), (uint64_t)plane * sizeof(float), 80u, (uint32_t)box_h,
                                (uint32_t)box_planes);
}

struct Arena {
    std::vector<void*> ptrs;
    size_t bytes = 0;
    template <typename T>
    int alloc(T** out, size_t count) {
        void* p = nullptr;
        size_t b = count * sizeof(T);
        if (b == 0) b = sizeof(T);
        cudaError_t e = cudaMalloc(&p, b);
        if (e != cudaSuccess) {
            set_error("cudaMalloc(%zu bytes) failed: %s", b, cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? MAVD_ERR_NOMEM : MAVD_ERR_CUDA;
        }
        ptrs.push_back(p);
        bytes += b;
        *out = (T*)p;
        return MAVD_OK;
    }
    template <typename T>
    int upload(T** out, const std::vector<T>& v) {
        int rc = alloc(out, v.size());
        if (rc != MAVD_OK) return rc;
        if (!v.empty()) MAVD_CUDA(cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
        return MAVD_OK;
    }
};

static int alloc_slot(Arena& A, mavd_handle_s::HostSlot& S, int F, int B, size_t npx) {
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

struct mavd_handle_full : mavd_handle_s {
    Arena arena;
};

static void drop_graphs(mavd_handle h);

// streams, events, graphs and pinned staging of a handle (everything but the device arena)
static void release_host_side(mavd_handle_full* H) {
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
    for (auto& r : H->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (cudaEvent_t e : H->prof.pool) cudaEventDestroy(e);
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
    mavd_handle_full* H = new (std::nothrow) mavd_handle_full();
    MAVD_REQUIRE(H != nullptr, MAVD_ERR_NOMEM, "out of host memory");
    H->cfg = *cfg;
    mavd_default_tuning(&H->tune);
    const mavd_farneback_params& fp = cfg->farneback;
    const int W = cfg->width, Hh = cfg->height, B = cfg->max_pairs;
    const int F = 2 * B;  // worst case: independent pairs
    H->max_frames = F;
    Arena& A = H->arena;
    int rc = MAVD_OK;
    auto fail = [&](int code) {
        for (void* p : A.ptrs) cudaFree(p);
        release_host_side(H);
        delete H;
        return code;
    };
#define C_TRY(x) do { rc = (x); if (rc != MAVD_OK) return fail(rc); } while (0)

    // level schedule (SURVEY §8 a2): levels = N -> up to N+1 images, 32-pixel cap
    int k = 0;
    double sc = 1.0;
    while (k < fp.levels) {
        sc *= fp.pyr_scale;
        if (W * sc < 32 || Hh * sc < 32) break;
        ++k;
    }
    if (k + 1 > kMaxLevels) {
        set_error("too many pyramid levels (%d)", k + 1);
        return fail(MAVD_ERR_UNSUPPORTED);
    }
    H->n_levels = k + 1;
    for (int li = 0; li < H->n_levels; ++li) {
        Level& L = H->lv[li];
        L.k = li;
        double s = 1.0;
        for (int i = 0; i < li; ++i) s *= fp.pyr_scale;
        L.scale = s;
        const double sigma = (1. / s - 1) * 0.5;
        L.sigma = (float)sigma;
        L.ksz = std::max(cv_round(sigma * 5) | 1, 3);
        L.w = cv_round(W * s);
        L.h = cv_round(Hh * s);
        L.pitch = round_up(L.w, 64);
        L.plane = (size_t)L.pitch * L.h;
        if (li > 0) {
            // combined blur + bilinear-resize filter per output sample: c_j = (1-a) k_j + a k_{j-1}
            const std::vector<float> kk = gaussian_kernel(L.ksz, sigma);
            const int taps = round_up(L.ksz + 1, 4), r = L.ksz / 2;   // zero padded to whole float4 groups
            for (int axis = 0; axis < 2; ++axis) {
                const int src = axis == 0 ? W : Hh, dst = axis == 0 ? L.w : L.h;
                std::vector<int> i0;
                std::vector<float> a;
                resize_tables(src, dst, i0, a);
                std::vector<int> base(dst);
                std::vector<float> tab((size_t)dst * taps);
                for (int d = 0; d < dst; ++d) {
                    base[d] = i0[d] - r;
                    for (int j = 0; j < taps; ++j) {
                        const float k0 = j < L.ksz ? kk[j] : 0.f, k1 = (j >= 1 && j <= L.ksz) ? kk[j - 1] : 0.f;
                        tab[(size_t)d * taps + j] = (1.f - a[d]) * k0 + a[d] * k1;
                    }
                }
                {
                    // pyr_scale 0.5 with src = dst * 2^li: the level is an exact decimation (farneback.cu: HalfPyr)
                    static const int kT[7] = {0, 4, 10, 20, 40, 80, 160}, kNB[7] = {0, 1, 3, 6, 12, 24, 48};
                    const int lc = std::min(li, 6);
                    bool half = li <= 6 && L.ksz + 1 == kT[lc] && dst >= 1 && src == dst << lc;
                    for (int d = 0; half && d < dst; ++d) {
                        half = base[d] == (d << lc) - kNB[lc];
                        for (int j = 0; half && j < taps; ++j) half = tab[(size_t)d * taps + j] == tab[j];
                    }
                    for (int j = kT[lc]; half && j < taps; ++j) half = tab[j] == 0.f;
                    (axis == 0 ? L.x_half : L.y_half) = half;
                    if (half) std::copy(tab.begin(), tab.begin() + kT[lc], axis == 0 ? L.xwt : L.ywt);
                }
                if (axis == 0) {
                    C_TRY(A.upload(&L.xbase, base)); C_TRY(A.upload(&L.xtab, tab));
                    std::vector<float> tabT((size_t)dst * taps);
                    for (int d = 0; d < dst; ++d)
                        for (int j = 0; j < taps; ++j) tabT[(size_t)j * dst + d] = tab[(size_t)d * taps + j];
                    C_TRY(A.upload(&L.xtabT, tabT));
                    L.hspan_max = 0;
                    L.hstride_min = dst > 1 ? src : 0;
                    for (int d0 = 0; d0 < dst; d0 += 64)
                        L.hspan_max = std::max(L.hspan_max, base[std::min(d0 + 63, dst - 1)] + taps - base[d0]);
                    for (int d = 1; d < dst; ++d) L.hstride_min = std::min(L.hstride_min, base[d] - base[d - 1]);
                }
                else           { C_TRY(A.upload(&L.ybase, base)); C_TRY(A.upload(&L.ytab, tab)); }
            }
            C_TRY(A.alloc(&L.tmp, (size_t)F * L.h * round_up(W, 4)));   // vertical-pass output [F][h_l][Wp]
        }
        C_TRY(A.alloc(&L.img, (size_t)F * L.plane));
        // polynomial expansion of the float levels: one TMA box {80, 32 + 2 poly_n} of the level image per tile
        L.has_tmap_img = li > 0 && make_plane_tensor_map(&L.tmapImg, L.img, L.pitch, L.h, F, L.plane, 32 + 2 * fp.poly_n, 1);
        C_TRY(A.alloc(&L.R, (size_t)F * 5 * L.plane));
        C_TRY(A.alloc(&L.M[0], (size_t)B * 5 * L.plane));
        C_TRY(A.alloc(&L.M[1], (size_t)B * 5 * L.plane));
        if (li > 0) C_TRY(A.alloc(&L.flow, (size_t)B * 2 * L.plane));
        // padded columns of R/M are read by vector loads of edge tiles: keep them finite
        cudaMemset(L.img, 0, (size_t)F * L.plane * sizeof(float));
        cudaMemset(L.R, 0, (size_t)F * 5 * L.plane * sizeof(float));
        cudaMemset(L.M[0], 0, (size_t)B * 5 * L.plane * sizeof(float));
        cudaMemset(L.M[1], 0, (size_t)B * 5 * L.plane * sizeof(float));
        const int m = fp.winsize / 2;
        if (m >= 5 && m <= 8)
            L.has_tmap = make_plane_tensor_map(&L.tmapM[0], L.M[0], L.pitch, L.h, B * 5, L.plane, 32 + 2 * m, 5) &&
                         make_plane_tensor_map(&L.tmapM[1], L.M[1], L.pitch, L.h, B * 5, L.plane, 32 + 2 * m, 5) &&
                         make_plane_tensor_map(&L.tmapR, L.R, L.pitch, L.h, F * 5, L.plane, 48, 10) &&
                         make_plane_tensor_map(&L.tmapRbox, L.R, L.pitch, L.h, F * 5, L.plane, 32 + 2 * m, 5);
        if (L.has_tmap)
            L.has_tmap16 = make_plane_tensor_map(&L.tmapM16[0], L.M[0], L.pitch, L.h, B * 5, L.plane, 16 + 2 * m, 5) &&
                           make_plane_tensor_map(&L.tmapM16[1], L.M[1], L.pitch, L.h, B * 5, L.plane, 16 + 2 * m, 5) &&
                           make_plane_tensor_map(&L.tmapRbox16, L.R, L.pitch, L.h, F * 5, L.plane, 16 + 2 * m, 5);
    }
    for (int li = 0; li + 1 < H->n_levels; ++li) {
        Level& L = H->lv[li];
        const Level& C = H->lv[li + 1];
        std::vector<int> i0;
        std::vector<float> a;
        resize_tables(C.w, L.w, i0, a);
        C_TRY(A.upload(&L.fxi0, i0));
        C_TRY(A.upload(&L.fxa, a));
        resize_tables(C.h, L.h, i0, a);
        C_TRY(A.upload(&L.fyi0, i0));
        C_TRY(A.upload(&L.fya, a));
    }
    C_TRY(poly_setup(fp.poly_n, fp.poly_sigma, H->poly));
    {
        // FarnebackUpdateFlow_GaussianBlur half kernel
        const int m = fp.winsize / 2;
        const double sigma = m * 0.3;
        std::vector<float> kf(m + 1);
        double s = 0;
        for (int i = 0; i <= m; ++i) {
            kf[i] = (float)exp(-i * i / (2 * sigma * sigma));
            s += (i == 0 ? 1.0 : 2.0) * kf[i];
        }
        for (int i = 0; i <= m; ++i) kf[i] = (float)(kf[i] * (1.0 / s));
        C_TRY(A.upload(&H->gauss_win, kf));
    }
    // detection workspace
    const size_t npx = (size_t)W * Hh;
    C_TRY(A.alloc(&H->d_imu, B));
    C_TRY(A.alloc(&H->d_foe, 2 * (size_t)B));
    C_TRY(A.alloc(&H->d_ninter, B));
    C_TRY(A.alloc(&H->d_labels, B * npx));
    C_TRY(A.alloc(&H->d_scan, B * npx + 2 * (size_t)B * (npx / 128 + 2) + 64));   // rank, unit counts, unit list (ccl_*)
    C_TRY(A.alloc(&H->d_total, B * npx));
    C_TRY(A.alloc(&H->d_fixed, B * npx));
    C_TRY(A.alloc(&H->d_flow, B * npx * 2));
    for (int k = 0; k < MAVD_HOST_SLOTS; ++k) {
        mavd_handle_s::HostSlot& S = H->slot[k];
        // slot 0 is always there (mavd_process_host); further slots appear on their first submit
        if (k == 0) C_TRY(alloc_slot(A, S, F, B, npx));
    }
    C_TRY(A.alloc(&H->d_stats_tmp, B));
    {
        // detector.py:90-91 evaluated with host IEEE doubles: division, subtraction, exact doubling
        std::vector<double> xn(W), yn(Hh);
        for (int x = 0; x < W; ++x) { volatile double q = (double)x / (double)W; volatile double d = q - 0.5; xn[x] = -d * 2.0; }
        for (int y = 0; y < Hh; ++y) { volatile double q = (double)y / (double)Hh; volatile double d = q - 0.5; yn[y] = -d * 2.0; }
        C_TRY(A.upload(&H->d_xn, xn));
        C_TRY(A.upload(&H->d_yn, yn));
    }
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
        cudaError_t e = cudaMallocHost((void**)&H->h_imu_ring, sizeof(mavd_imu) * mavd_handle_s::kImuRing * (size_t)B);
        for (int k = 0; e == cudaSuccess && k < mavd_handle_s::kImuRing; ++k)
            e = cudaEventCreateWithFlags(&H->imu_ev[k], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            set_error("imu staging: %s", cudaGetErrorString(e));
            return fail(e == cudaErrorMemoryAllocation ? MAVD_ERR_NOMEM : MAVD_ERR_CUDA);
        }
    }
    H->bytes = A.bytes;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error("device error during create: %s", cudaGetErrorString(e));
        return fail(MAVD_ERR_CUDA);
    }
    *out = H;
    return MAVD_OK;
#undef C_TRY
}

int mavd_destroy(mavd_handle h) {
    if (!h) return MAVD_OK;
    mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
    DeviceGuard dg(H->cfg.device);
    cudaDeviceSynchronize();
    for (void* p : H->arena.ptrs) cudaFree(p);
    release_host_side(H);
    delete H;
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
    *out = h->bytes;
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

// taps read "the last mavd_farneback call": recorded here, outside the (possibly replayed) launch sequence
static void note_farneback_call(mavd_handle h, const uint8_t* d_frames, int n_pairs, int pair_stride, float* d_flow) {
    h->last_pairs = n_pairs;
    h->last_stride = pair_stride;
    h->last_flow0 = d_flow;
    h->last_frames = d_frames;
}

int mavd_farneback_tap(mavd_handle h, int32_t kind, int32_t level, int32_t index, float* d_out, void* stream) {
    MAVD_REQUIRE(h && d_out, MAVD_ERR_INVALID, "tap: NULL argument");
    DeviceGuard dg(h->cfg.device);
    MAVD_REQUIRE(index >= 0 && index < h->max_frames, MAVD_ERR_INVALID, "tap: index out of range");
    return farneback_tap(h, kind, level, index, d_out, (cudaStream_t)stream);
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
    mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
    TRY(H->arena.alloc(&H->d_det_area, (size_t)h->cfg.max_pairs * det_lab_stride(h)));
    TRY(H->arena.alloc(&H->d_det_nlabels, (size_t)h->cfg.max_pairs));
    H->bytes = H->arena.bytes;
    return MAVD_OK;
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

// The corner workspace of mavd::gftt_chunk() frames, carved from one allocation made by the first corner call.
static GfttWork gftt_work(mavd_handle h) {
    const int W = h->cfg.width, Hh = h->cfg.height, G = gftt_chunk();
    const size_t npx = (size_t)W * Hh;
    char* p = (char*)h->sp_gftt;
    GfttWork w;
    w.rows = (double*)p;                  p += sizeof(double) * 3 * npx * G;
    w.keys = (unsigned long long*)p;      p += sizeof(unsigned long long) * gftt_key_cap(W, Hh) * G;
    w.cov = (float3*)p;                   p += sizeof(float3) * npx * G;
    w.eig = (float*)p;                    p += sizeof(float) * npx * G;
    w.grid = (int*)p;                     p += sizeof(int) * gftt_grid_cap(W, Hh) * G;
    w.maxv = (uint32_t*)p;                p += sizeof(uint32_t) * G;
    w.n_cand = (int*)p;
    return w;
}

static size_t gftt_work_bytes(mavd_handle h) {
    const int W = h->cfg.width, Hh = h->cfg.height, G = gftt_chunk();
    const size_t npx = (size_t)W * Hh;
    return (sizeof(double) * 3 * npx + sizeof(unsigned long long) * gftt_key_cap(W, Hh) + sizeof(float3) * npx +
            sizeof(float) * npx + sizeof(int) * gftt_grid_cap(W, Hh) + sizeof(uint32_t) + sizeof(int)) * G;
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
    if (!h->sp_gftt) {
        mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
        char* base = nullptr;
        TRY(H->arena.alloc(&base, gftt_work_bytes(h)));
        H->sp_gftt = base;
        H->bytes = H->arena.bytes;
    }
    return gftt_run(h, gftt_work(h), d_frames, n_frames, p, d_mask, d_mask ? mask_stride : 0, d_corners, d_count, d_eig,
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
    if (!h->sp_pyr) {
        mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
        const int W = h->cfg.width, Hh = h->cfg.height;
        uint8_t* pyr = nullptr;
        short2* der = nullptr;
        TRY(H->arena.alloc(&pyr, (size_t)h->max_frames * lk_pyr_frame_bytes(W, Hh)));
        TRY(H->arena.alloc(&der, (size_t)h->max_frames * lk_der_frame_elems(W, Hh)));
        H->sp_pyr = pyr;
        H->sp_der = der;
        H->bytes = H->arena.bytes;
    }
    return lk_run(h, h->sp_pyr, h->sp_der, d_frames, n_pairs, pair_stride, p, d_prev_pts, n_points, d_n_points,
                  d_next_pts, d_status, d_err, (cudaStream_t)stream);
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

int mavd_detect_det(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
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

int mavd_detect_ex(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                   const int32_t* d_samples, const mavd_aux_inputs* d_aux, uint8_t* d_total_out, uint8_t* d_fixed_out,
                   mavd_frame_record* d_records, void* stream) {
    return mavd_detect_det(h, d_flow, n, h_imu, prm, d_samples, d_aux, d_total_out, d_fixed_out, d_records, 0, nullptr,
                           stream);
}

int mavd_detect(mavd_handle h, const float* d_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                const int32_t* d_samples, const uint8_t* d_sky, int64_t sky_stride, const uint8_t* d_seg,
                int64_t seg_stride, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                void* stream) {
    const mavd_aux_inputs aux = {d_sky, sky_stride, d_seg, seg_stride, nullptr};
    return mavd_detect_ex(h, d_flow, n, h_imu, prm, d_samples, &aux, d_total_out, d_fixed_out, d_records, stream);
}

int mavd_process_det(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                     const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                     float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                     int32_t max_det, mavd_detection* d_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n_pairs, "process"));
    MAVD_REQUIRE(pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    TRY(check_det(h, max_det, d_det, "process"));
    if (!d_det) max_det = 0;
    if (n_pairs == 0) return MAVD_OK;
    MAVD_REQUIRE(d_frames && d_samples && d_records, MAVD_ERR_INVALID, "process: NULL buffer");
    StreamScope ss(h, stream);
    mavd_detect_params p;
    if (prm) p = *prm; else mavd_default_detect_params(&p);
    const mavd_aux_inputs aux = d_aux ? *d_aux : kNoAux;
    float* flow = d_flow_out ? d_flow_out : h->d_flow;
    uint8_t* fixed = d_fixed_out ? d_fixed_out : h->d_fixed;
    int n64 = 0, n32 = 0;
    TRY(upload_imu(h, h_imu, n_pairs, ss.s, &n64, &n32));
    note_farneback_call(h, d_frames, n_pairs, pair_stride, flow);
    return run_graphed(h, std::move(KeyBuilder()(int64_t(3))(d_frames)(int64_t(n_pairs))(int64_t(pair_stride))(p)(int64_t(n64))(int64_t(h->batch_rot > 0))
                                        (int64_t(n32))(d_samples)(aux)(flow)(d_total_out)(fixed)(d_records)(int64_t(max_det))
                                        (d_det).k),
                       ss.s, [&](cudaStream_t s) {
                           TRY(farneback_run(h, d_frames, n_pairs, pair_stride, flow, s));
                           return detect_run(h, flow, n_pairs, p, n64, n32, d_samples, aux, d_total_out, fixed, d_records,
                                             max_det, d_det, s);
                       });
}

int mavd_process_ex(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                    const mavd_detect_params* prm, const int32_t* d_samples, const mavd_aux_inputs* d_aux,
                    float* d_flow_out, uint8_t* d_total_out, uint8_t* d_fixed_out, mavd_frame_record* d_records,
                    void* stream) {
    return mavd_process_det(h, d_frames, n_pairs, pair_stride, h_imu, prm, d_samples, d_aux, d_flow_out, d_total_out,
                            d_fixed_out, d_records, 0, nullptr, stream);
}

int mavd_process(mavd_handle h, const uint8_t* d_frames, int32_t n_pairs, int32_t pair_stride, const mavd_imu* h_imu,
                 const mavd_detect_params* prm, const int32_t* d_samples, const uint8_t* d_sky, int64_t sky_stride,
                 const uint8_t* d_seg, int64_t seg_stride, float* d_flow_out, uint8_t* d_total_out,
                 uint8_t* d_fixed_out, mavd_frame_record* d_records, void* stream) {
    const mavd_aux_inputs aux = {d_sky, sky_stride, d_seg, seg_stride, nullptr};
    return mavd_process_ex(h, d_frames, n_pairs, pair_stride, h_imu, prm, d_samples, &aux, d_flow_out, d_total_out,
                           d_fixed_out, d_records, stream);
}

// ------------------------------------------------------------------------------------------------
// Host-buffer calls: three-stage pipeline over MAVD_HOST_SLOTS staging sets (copy-in stream, the caller's compute
// stream, copy-out stream).
// ------------------------------------------------------------------------------------------------
static int ensure_slot(mavd_handle h, int slot, bool want_flow_out, bool want_flow_in, bool want_bits_in, bool want_bits_out,
                       bool want_gt, bool want_det) {
    mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
    mavd_handle_s::HostSlot& S = H->slot[slot];
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
    const int B = h->cfg.max_pairs;
    if (!S.d_frames) TRY(alloc_slot(H->arena, S, h->max_frames, B, npx));
    if (want_flow_out && !S.d_flow) TRY(H->arena.alloc(&S.d_flow, B * npx * 2));
    if (want_flow_in && !S.d_flow_in) TRY(H->arena.alloc(&S.d_flow_in, B * npx * 2));
    if (want_bits_in && !S.d_bits_in) TRY(H->arena.alloc(&S.d_bits_in, 2 * B * pb));
    if (want_bits_out && !S.d_bits_out) TRY(H->arena.alloc(&S.d_bits_out, B * pb));
    if (want_gt && !S.d_gt_flow) TRY(H->arena.alloc(&S.d_gt_flow, B * npx * 2));
    if (want_det && !S.d_det) TRY(H->arena.alloc(&S.d_det, (size_t)B * MAVD_MAX_DETECTIONS));
    if (!H->s_in) MAVD_CUDA(cudaStreamCreateWithFlags(&H->s_in, cudaStreamNonBlocking));
    if (!H->s_out) MAVD_CUDA(cudaStreamCreateWithFlags(&H->s_out, cudaStreamNonBlocking));
    H->bytes = H->arena.bytes;
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

int mavd_submit_host_det(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                         const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                         const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                         mavd_frame_record* h_records, int32_t max_det, mavd_detection* h_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n_pairs, "submit_host"));
    if (h_det)
        MAVD_REQUIRE(max_det >= 1 && max_det <= MAVD_MAX_DETECTIONS, MAVD_ERR_INVALID,
                     "submit_host: max_det %d outside 1..%d", max_det, MAVD_MAX_DETECTIONS);
    MAVD_REQUIRE(slot >= 0 && slot < MAVD_HOST_SLOTS, MAVD_ERR_INVALID, "slot %d out of range", slot);
    MAVD_REQUIRE(pair_stride == 1 || pair_stride == 2, MAVD_ERR_INVALID, "pair_stride must be 1 or 2");
    MAVD_REQUIRE(n_pairs >= 1, MAVD_ERR_INVALID, "submit_host: empty batch");
    MAVD_REQUIRE(h_frames && h_samples && h_records, MAVD_ERR_INVALID, "submit_host: NULL buffer");
    const mavd_aux_inputs ha = h_aux ? *h_aux : kNoAux;
    TRY(check_aux_strides(h, ha, flags));
    TRY(check_samples(h_samples, n_pairs, h->cfg.width, h->cfg.height));
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
    const bool bgr = (flags & MAVD_HOST_BGR) != 0, fixed_packed = (flags & MAVD_HOST_FIXED_PACKED) != 0;
    TRY(ensure_slot(h, slot, h_flow_out != nullptr, false, (flags & (MAVD_HOST_SEG_PACKED | MAVD_HOST_SKY_PACKED)) != 0,
                    fixed_packed && h_fixed_out, ha.gt_flow != nullptr, h_det != nullptr));
    mavd_handle_s::HostSlot& S = h->slot[slot];
    MAVD_REQUIRE(!S.busy, MAVD_ERR_INVALID, "slot %d is still in flight: call mavd_wait_host first", slot);
    const int n_frames = pair_stride == 1 ? n_pairs + 1 : 2 * n_pairs;
    if (bgr && !S.d_bgr) {
        mavd_handle_full* H = static_cast<mavd_handle_full*>(h);
        TRY(H->arena.alloc(&S.d_bgr, (size_t)h->max_frames * npx * 3));
        H->bytes = H->arena.bytes;
    }
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
        TRY(mavd_process_det(h, S.d_frames, n_pairs, pair_stride, h_imu, prm, S.d_samples, &da,
                             h_flow_out ? S.d_flow : nullptr, nullptr, S.d_fixed, S.d_records, max_det,
                             h_det ? S.d_det : nullptr, s));
    MAVD_CUDA(cudaEventRecord(S.ev_done, s));
    // copy-out stream
    MAVD_CUDA(cudaStreamWaitEvent(h->s_out, S.ev_done, 0));
    MAVD_CUDA(cudaMemcpyAsync(h_records, S.d_records, sizeof(mavd_frame_record) * n_pairs, cudaMemcpyDeviceToHost, h->s_out));
    if (h_fixed_out && fixed_packed) {
        TRY(pack_mask_run(S.d_fixed, n_pairs, (int64_t)npx, S.d_bits_out, h->s_out));
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_bits_out, pb * n_pairs, cudaMemcpyDeviceToHost, h->s_out));
    } else if (h_fixed_out) {
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_fixed, npx * n_pairs, cudaMemcpyDeviceToHost, h->s_out));
    }
    if (h_flow_out)
        MAVD_CUDA(cudaMemcpyAsync(h_flow_out, S.d_flow, sizeof(float) * 2 * npx * n_pairs, cudaMemcpyDeviceToHost, h->s_out));
    if (h_det)
        MAVD_CUDA(cudaMemcpyAsync(h_det, S.d_det, sizeof(mavd_detection) * max_det * n_pairs, cudaMemcpyDeviceToHost,
                                  h->s_out));
    MAVD_CUDA(cudaEventRecord(S.ev_out, h->s_out));
    // the next batch's copy-in must not overwrite staging a kernel still reads: ordered by slot reuse rule
    S.busy = true;
    return MAVD_OK;
}

int mavd_submit_host_ex(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                        const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                        const mavd_aux_inputs* h_aux, int32_t flags, float* h_flow_out, uint8_t* h_fixed_out,
                        mavd_frame_record* h_records, void* stream) {
    return mavd_submit_host_det(h, slot, h_frames, n_pairs, pair_stride, h_imu, prm, h_samples, h_aux, flags, h_flow_out,
                                h_fixed_out, h_records, 0, nullptr, stream);
}

int mavd_submit_host(mavd_handle h, int32_t slot, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                     const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                     const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                     float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream) {
    const mavd_aux_inputs aux = {h_sky, sky_stride, h_seg, seg_stride, nullptr};
    return mavd_submit_host_ex(h, slot, h_frames, n_pairs, pair_stride, h_imu, prm, h_samples, &aux, 0, h_flow_out,
                               h_fixed_out, h_records, stream);
}

int mavd_submit_host_bgr(mavd_handle h, int32_t slot, const uint8_t* h_bgr_frames, int32_t n_pairs, int32_t pair_stride,
                         const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                         const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                         float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream) {
    const mavd_aux_inputs aux = {h_sky, sky_stride, h_seg, seg_stride, nullptr};
    return mavd_submit_host_ex(h, slot, h_bgr_frames, n_pairs, pair_stride, h_imu, prm, h_samples, &aux, MAVD_HOST_BGR,
                               h_flow_out, h_fixed_out, h_records, stream);
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

int mavd_process_host(mavd_handle h, const uint8_t* h_frames, int32_t n_pairs, int32_t pair_stride,
                      const mavd_imu* h_imu, const mavd_detect_params* prm, const int32_t* h_samples,
                      const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg, int64_t seg_stride,
                      float* h_flow_out, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n_pairs, "process_host"));
    if (n_pairs == 0) return MAVD_OK;
    TRY(mavd_wait_host(h, 0));
    TRY(mavd_submit_host(h, 0, h_frames, n_pairs, pair_stride, h_imu, prm, h_samples, h_sky, sky_stride, h_seg,
                         seg_stride, h_flow_out, h_fixed_out, h_records, stream));
    return mavd_wait_host(h, 0);
}

int mavd_detect_host_det(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                         const mavd_detect_params* prm, const int32_t* h_samples, const mavd_aux_inputs* h_aux,
                         int32_t flags, uint8_t* h_fixed_out, mavd_frame_record* h_records, int32_t max_det,
                         mavd_detection* h_det, void* stream) {
    DeviceGuard dg(h ? h->cfg.device : -1);
    TRY(check_batch(h, n, "detect_host"));
    if (h_det)
        MAVD_REQUIRE(max_det >= 1 && max_det <= MAVD_MAX_DETECTIONS, MAVD_ERR_INVALID,
                     "detect_host: max_det %d outside 1..%d", max_det, MAVD_MAX_DETECTIONS);
    if (n == 0) return MAVD_OK;
    MAVD_REQUIRE(h_flow && h_samples && h_records, MAVD_ERR_INVALID, "detect_host: NULL buffer");
    MAVD_REQUIRE((flags & MAVD_HOST_BGR) == 0, MAVD_ERR_INVALID, "detect_host: MAVD_HOST_BGR has no meaning here");
    const mavd_aux_inputs ha = h_aux ? *h_aux : kNoAux;
    TRY(check_aux_strides(h, ha, flags));
    TRY(check_samples(h_samples, n, h->cfg.width, h->cfg.height));
    const size_t npx = (size_t)h->cfg.width * h->cfg.height;
    const size_t pb = (size_t)packed_mask_bytes((int64_t)npx);
    const bool fixed_packed = (flags & MAVD_HOST_FIXED_PACKED) != 0;
    TRY(mavd_wait_host(h, 0));
    TRY(ensure_slot(h, 0, false, true, (flags & (MAVD_HOST_SEG_PACKED | MAVD_HOST_SKY_PACKED)) != 0,
                    fixed_packed && h_fixed_out, ha.gt_flow != nullptr, h_det != nullptr));
    mavd_handle_s::HostSlot& S = h->slot[0];
    StreamScope ss(h, stream);
    cudaStream_t s = ss.s;
    MAVD_CUDA(cudaMemcpyAsync(S.d_flow_in, h_flow, sizeof(float) * 2 * npx * n, cudaMemcpyHostToDevice, s));
    MAVD_CUDA(cudaMemcpyAsync(S.d_samples, h_samples, sizeof(int32_t) * MAVD_SAMPLES_PER_FRAME * n, cudaMemcpyHostToDevice, s));
    mavd_aux_inputs da;
    TRY(stage_aux(h, S, ha, flags, n, s, &da));
    if (!(flags & MAVD_HOST_COPY_ONLY))
        TRY(mavd_detect_det(h, S.d_flow_in, n, h_imu, prm, S.d_samples, &da, nullptr, S.d_fixed, S.d_records, max_det,
                            h_det ? S.d_det : nullptr, s));
    MAVD_CUDA(cudaMemcpyAsync(h_records, S.d_records, sizeof(mavd_frame_record) * n, cudaMemcpyDeviceToHost, s));
    if (h_det)
        MAVD_CUDA(cudaMemcpyAsync(h_det, S.d_det, sizeof(mavd_detection) * max_det * n, cudaMemcpyDeviceToHost, s));
    if (h_fixed_out && fixed_packed) {
        TRY(pack_mask_run(S.d_fixed, n, (int64_t)npx, S.d_bits_out, s));
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_bits_out, pb * n, cudaMemcpyDeviceToHost, s));
    } else if (h_fixed_out) {
        MAVD_CUDA(cudaMemcpyAsync(h_fixed_out, S.d_fixed, npx * n, cudaMemcpyDeviceToHost, s));
    }
    MAVD_CUDA(cudaStreamSynchronize(s));
    return MAVD_OK;
}

int mavd_detect_host_ex(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu,
                        const mavd_detect_params* prm, const int32_t* h_samples, const mavd_aux_inputs* h_aux,
                        int32_t flags, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream) {
    return mavd_detect_host_det(h, h_flow, n, h_imu, prm, h_samples, h_aux, flags, h_fixed_out, h_records, 0, nullptr,
                                stream);
}

int mavd_detect_host(mavd_handle h, const float* h_flow, int32_t n, const mavd_imu* h_imu, const mavd_detect_params* prm,
                     const int32_t* h_samples, const uint8_t* h_sky, int64_t sky_stride, const uint8_t* h_seg,
                     int64_t seg_stride, uint8_t* h_fixed_out, mavd_frame_record* h_records, void* stream) {
    const mavd_aux_inputs aux = {h_sky, sky_stride, h_seg, seg_stride, nullptr};
    return mavd_detect_host_ex(h, h_flow, n, h_imu, prm, h_samples, &aux, 0, h_fixed_out, h_records, stream);
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
