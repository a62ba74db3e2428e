// Derotation, Focus-of-Expansion RANSAC, radial residual / masks / metrics and connected components
// for sm_100a.  Follows /root/reference/src/detector.py:70-117, focus_of_expansion.py:32-86,150-184,
// processor.py:306-362, im_helpers.py:55-84,244-252, utils.py:183-197 (SURVEY.md §8 a8-a14, a17).
//
// Parity-critical float64 arithmetic uses the explicit round-to-nearest intrinsics (__dmul_rn,
// __dadd_rn, ...) so that nvcc cannot contract a*b+c into an FMA: NumPy evaluates every ufunc with
// one rounding per operation and the masks must be bit-exact.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace mavd {

// ------------------------------------------------------------------------------------------------
// BGR -> gray: cv2.cvtColor(COLOR_BGR2GRAY) on uint8 == (B*3735 + G*19235 + R*9798 + 16384) >> 15
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bgr2gray_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray,
                                                      int64_t n) {
    int64_t i4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= n) return;
    if (i4 + 4 <= n && ((uintptr_t)bgr & 3) == 0 && ((uintptr_t)gray & 3) == 0) {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(bgr + i4 * 3);
        uint32_t a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
        uint8_t v[12];
        v[0] = a; v[1] = a >> 8; v[2] = a >> 16; v[3] = a >> 24;
        v[4] = b; v[5] = b >> 8; v[6] = b >> 16; v[7] = b >> 24;
        v[8] = c; v[9] = c >> 8; v[10] = c >> 16; v[11] = c >> 24;
        uint32_t out = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t g = (v[3 * k] * 3735u + v[3 * k + 1] * 19235u + v[3 * k + 2] * 9798u + 16384u) >> 15;
            out |= g << (8 * k);
        }
        *reinterpret_cast<uint32_t*>(gray + i4) = out;
    } else {
        for (int64_t i = i4; i < n && i < i4 + 4; ++i)
            gray[i] = (uint8_t)((bgr[3 * i] * 3735u + bgr[3 * i + 1] * 19235u + bgr[3 * i + 2] * 9798u + 16384u) >> 15);
    }
}

int bgr2gray_run(const uint8_t* d_bgr, uint8_t* d_gray, int64_t n, cudaStream_t s) {
    int64_t threads = (n + 3) / 4;
    bgr2gray_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(d_bgr, d_gray, n);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Derotation (detector.py:88-101), evaluated with NumPy's operation order, one rounding per op.
// ------------------------------------------------------------------------------------------------
struct Derot {
    double o0, o1, o2;  // omega = ang / dt
    double s0, s1;      // w*dt/2, h*dt/2
    double w, h;
    int on;
};

__device__ __forceinline__ Derot make_derot(const mavd_imu& imu, int w, int h) {
    Derot d;
    d.on = imu.derotate;
    d.o0 = __ddiv_rn(imu.ang[0], imu.dt);
    d.o1 = __ddiv_rn(imu.ang[1], imu.dt);
    d.o2 = __ddiv_rn(imu.ang[2], imu.dt);
    d.s0 = __ddiv_rn(__dmul_rn((double)w, imu.dt), 2.0);
    d.s1 = __ddiv_rn(__dmul_rn((double)h, imu.dt), 2.0);
    d.w = (double)w;
    d.h = (double)h;
    return d;
}

__device__ __forceinline__ void derot_at(const Derot& d, int x, int y, double& r0, double& r1) {
    const double xn = __dmul_rn(-__dsub_rn(__ddiv_rn((double)x, d.w), 0.5), 2.0);
    const double yn = __dmul_rn(-__dsub_rn(__ddiv_rn((double)y, d.h), 0.5), 2.0);
    // +o0*xn*yn - o1*xn**2 - o1 + o2*yn
    double t = __dmul_rn(__dmul_rn(d.o0, xn), yn);
    t = __dsub_rn(t, __dmul_rn(d.o1, __dmul_rn(xn, xn)));
    t = __dsub_rn(t, d.o1);
    t = __dadd_rn(t, __dmul_rn(d.o2, yn));
    r0 = __dmul_rn(t, d.s0);
    // -o2*xn + o0 + o0*yn**2 - o1*xn*yn
    double u = __dmul_rn(-d.o2, xn);
    u = __dadd_rn(u, d.o0);
    u = __dadd_rn(u, __dmul_rn(d.o0, __dmul_rn(yn, yn)));
    u = __dsub_rn(u, __dmul_rn(__dmul_rn(d.o1, xn), yn));
    r1 = __dmul_rn(u, d.s1);
}

template <typename T2>
__global__ void __launch_bounds__(256) derotate_kernel(const T2* __restrict__ flow, const mavd_imu* __restrict__ imu,
                                                      int w, int h, double2* __restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    if (x >= w) return;
    const Derot d = make_derot(imu[f], w, h);
    const size_t o = ((size_t)f * h + y) * w + x;
    const T2 v = flow[o];
    double r0 = 0.0, r1 = 0.0;
    if (d.on) derot_at(d, x, y, r0, r1);
    out[o] = make_double2(d.on ? __dsub_rn((double)v.x, r0) : (double)v.x,
                          d.on ? __dsub_rn((double)v.y, r1) : (double)v.y);
}

int derotate_run(mavd_handle H, const void* d_flow, int flow_is_f64, int n, const mavd_imu* d_imu, double* d_out,
                 cudaStream_t s) {
    dim3 g(ceil_div(H->cfg.width, 256), H->cfg.height, n);
    if (flow_is_f64)
        derotate_kernel<double2><<<g, 256, 0, s>>>((const double2*)d_flow, d_imu, H->cfg.width, H->cfg.height, (double2*)d_out);
    else
        derotate_kernel<float2><<<g, 256, 0, s>>>((const float2*)d_flow, d_imu, H->cfg.width, H->cfg.height, (double2*)d_out);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// FoE: 1000 flow-line intersections + consensus scoring.  One 1024-thread CTA per frame.
//   phase A  thread i builds intersection i (float64, utils.line_intersection order of operations)
//   phase B  order-preserving compaction of rows with x != 0 (ballot + warp offsets)
//   phase C  thread i counts estimates within ransac_threshold of estimate i
//   phase D  arg-max with first-maximum tie-break (warp shuffles, then across warps)
// sqrt(s) < T is evaluated as s < s*, s* = the smallest double whose correctly rounded square root
// is >= T (computed on the host), which is exactly equivalent and saves 10^6 double square roots.
// ------------------------------------------------------------------------------------------------
constexpr int kNP = MAVD_N_SAMPLE_PAIRS;

// kind 0: float32 flow, per-frame imu (derotation applied inline); 1: float32 flow as given;
// 2: float64 flow as given (get_FOE_dense on an already derotated field)
__global__ void __launch_bounds__(1024) foe_kernel(const void* __restrict__ flow, int kind,
                                                  const mavd_imu* __restrict__ imu,
                                                  const int32_t* __restrict__ samples, int w, int h,
                                                  double mag_thr, double sq_thr, double* __restrict__ foe,
                                                  int32_t* __restrict__ ninter) {
    pdl_entry();
    __shared__ double2 E[kNP];
    __shared__ int warp_cnt[32];
    __shared__ unsigned long long warp_best[32];
    const int f = blockIdx.x, i = threadIdx.x, lane = i & 31, wid = i >> 5;
    Derot d;
    d.on = 0;
    if (kind == 0) d = make_derot(imu[f], w, h);
    const int32_t* sm = samples + (size_t)f * MAVD_SAMPLES_PER_FRAME;

    bool valid = false;
    double ex = 0.0, ey = 0.0;
    if (i < kNP) {
        // indices are the caller's np.random.randint draws; a stale or wrong-resolution table must not read out of bounds
        const int y1 = min(max(sm[i], 0), h - 1), y2 = min(max(sm[i + kNP], 0), h - 1);
        const int x1 = min(max(sm[2 * kNP + i], 0), w - 1), x2 = min(max(sm[3 * kNP + i], 0), w - 1);
        float2 a = make_float2(0.f, 0.f), b = a;
        double f1x, f1y, f2x, f2y;
        bool keep;
        if (kind == 2) {
            const double2* fl = reinterpret_cast<const double2*>(flow) + (size_t)f * w * h;
            const double2 a2 = fl[(size_t)y1 * w + x1], b2 = fl[(size_t)y2 * w + x2];
            f1x = a2.x; f1y = a2.y; f2x = b2.x; f2y = b2.y;
            const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(f2x, f2x), __dmul_rn(f2y, f2y)));
            keep = !(mag < mag_thr);
        } else {
            const float2* fl = reinterpret_cast<const float2*>(flow) + (size_t)f * w * h;
            a = fl[(size_t)y1 * w + x1];
            b = fl[(size_t)y2 * w + x2];
        }
        if (kind == 2) {
        } else if (d.on) {
            double r0, r1;
            derot_at(d, x1, y1, r0, r1);
            f1x = __dsub_rn((double)a.x, r0); f1y = __dsub_rn((double)a.y, r1);
            derot_at(d, x2, y2, r0, r1);
            f2x = __dsub_rn((double)b.x, r0); f2y = __dsub_rn((double)b.y, r1);
            const double mag = __dsqrt_rn(__dadd_rn(__dmul_rn(f2x, f2x), __dmul_rn(f2y, f2y)));
            keep = !(mag < mag_thr);
        } else {
            f1x = a.x; f1y = a.y; f2x = b.x; f2y = b.y;
            const float mag = __fsqrt_rn(__fadd_rn(__fmul_rn(b.x, b.x), __fmul_rn(b.y, b.y)));
            keep = !(mag < (float)mag_thr);
        }
        if (keep) {
            const double cx1 = x1, cy1 = y1, cx2 = x2, cy2 = y2;
            const double p1x = __dadd_rn(f1x, cx1), p1y = __dadd_rn(f1y, cy1);
            const double p2x = __dadd_rn(f2x, cx2), p2y = __dadd_rn(f2y, cy2);
            const double xd0 = __dsub_rn(cx1, p1x), xd1 = __dsub_rn(cx2, p2x);
            const double yd0 = __dsub_rn(cy1, p1y), yd1 = __dsub_rn(cy2, p2y);
            const double div = __dsub_rn(__dmul_rn(xd0, yd1), __dmul_rn(xd1, yd0));
            if (div != 0.0) {
                const double d0 = __dsub_rn(__dmul_rn(cx1, p1y), __dmul_rn(cy1, p1x));
                const double d1 = __dsub_rn(__dmul_rn(cx2, p2y), __dmul_rn(cy2, p2x));
                ex = __ddiv_rn(__dsub_rn(__dmul_rn(d0, xd1), __dmul_rn(d1, xd0)), div);
                ey = __ddiv_rn(__dsub_rn(__dmul_rn(d0, yd1), __dmul_rn(d1, yd0)), div);
                valid = (ex != 0.0);  // also true for NaN, as in NumPy
            }
        }
    }
    // ---- phase B ----
    const unsigned bal = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) warp_cnt[wid] = __popc(bal);
    __syncthreads();
    if (wid == 0) {
        int v = warp_cnt[lane], incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        warp_cnt[lane] = incl - v;
        if (lane == 31) warp_best[0] = (unsigned long long)incl;  // total, parked here for a moment
    }
    __syncthreads();
    const int K = (int)warp_best[0];
    if (valid) E[warp_cnt[wid] + __popc(bal & ((1u << lane) - 1u))] = make_double2(ex, ey);
    __syncthreads();
    // ---- phase C ----
    int score = -1;
    if (i < K) {
        const double2 me = E[i];
        int cnt = 0;
        for (int j = 0; j < K; ++j) {
            const double2 o = E[j];
            const double dx = __dsub_rn(o.x, me.x), dy = __dsub_rn(o.y, me.y);
            const double s2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            cnt += (s2 < sq_thr) ? 1 : 0;
        }
        score = cnt - 1;
    }
    // ---- phase D: maximise (score, -index) ----
    unsigned long long key = (score > 0) ? (((unsigned long long)(unsigned)score << 32) | (unsigned)(0x7fffffff - i)) : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(0xffffffffu, key, o);
        key = t > key ? t : key;
    }
    __syncthreads();
    if (lane == 0) warp_best[wid] = key;
    __syncthreads();
    if (wid == 0) {
        key = warp_best[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long t = __shfl_xor_sync(0xffffffffu, key, o);
            key = t > key ? t : key;
        }
        if (lane == 0) {
            double bx = 0.0, by = 0.0;
            if (key != 0ull) {
                const int best = 0x7fffffff - (int)(key & 0xffffffffu);
                bx = E[best].x;
                by = E[best].y;
            }
            foe[2 * f] = bx;
            foe[2 * f + 1] = by;
            ninter[f] = K;
        }
    }
}

// smallest double s with correctly-rounded sqrt(s) >= T  (so that  sqrt(s) < T  <=>  s < s*)
static double sqrt_threshold(double T) {
    if (!(T > 0.0)) return 0.0;
    double s = T * T;
    while (sqrt(s) >= T) s = nextafter(s, 0.0);
    while (sqrt(s) < T) s = nextafter(s, INFINITY);
    return s;
}

int foe_run(mavd_handle H, const void* d_flow, int flow_kind, int n, const mavd_imu* d_imu,
            const mavd_detect_params& prm, const int32_t* d_samples, double* d_foe, int32_t* d_ninter, cudaStream_t s) {
    ProfScope ps(&H->prof, MAVD_PROF_FOE, s);
    MAVD_CUDA(launch_chained(pdl_next(H), foe_kernel, n, 1024, 0, s, d_flow, flow_kind, d_imu, d_samples, H->cfg.width,
                             H->cfg.height, prm.magnitude_threshold, sqrt_threshold(prm.ransac_threshold), d_foe, d_ninter));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// FocusOfExpansion.ransac on a caller-supplied (K, 2) float64 array (focus_of_expansion.py:32-54):
// one CTA, thread i scores estimates i, i + 1024, ...; first strict maximum wins.
__global__ void __launch_bounds__(1024) ransac_kernel(const double2* __restrict__ E, int K, double sq_thr,
                                                     double* __restrict__ out) {
    __shared__ unsigned long long warp_best[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long key = 0ull;
    for (int i = threadIdx.x; i < K; i += 1024) {
        const double2 me = E[i];
        int cnt = 0;
        for (int j = 0; j < K; ++j) {
            const double2 o = __ldg(E + j);
            const double dx = __dsub_rn(o.x, me.x), dy = __dsub_rn(o.y, me.y);
            cnt += (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < sq_thr) ? 1 : 0;
        }
        const int score = cnt - 1;
        const unsigned long long k = (score > 0) ? (((unsigned long long)(unsigned)score << 32) | (unsigned)(0x7fffffff - i)) : 0ull;
        key = k > key ? k : key;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, key, o);
        key = t > key ? t : key;
    }
    if (lane == 0) warp_best[wid] = key;
    __syncthreads();
    if (wid == 0) {
        key = warp_best[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, key, o);
            key = t > key ? t : key;
        }
        if (lane == 0) {
            double bx = 0.0, by = 0.0;
            if (key != 0ull) {
                const int best = 0x7fffffff - (int)(key & 0xffffffffu);
                bx = E[best].x;
                by = E[best].y;
            }
            out[0] = bx;
            out[1] = by;
        }
    }
}

int ransac_run(const double* d_estimates, int K, double threshold, double* d_out, cudaStream_t s) {
    ransac_kernel<<<1, 1024, 0, s>>>((const double2*)d_estimates, K, sqrt_threshold(threshold), d_out);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

__global__ void gather_max_phi_kernel(const char* stats_base, size_t stats_stride, int n, double* out) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < n) out[f] = reinterpret_cast<const mavd_frame_stats*>(stats_base + (size_t)f * stats_stride)->max_phi;
}

int gather_max_phi_run(const mavd_frame_stats* d_stats, int n, double* d_out, cudaStream_t s) {
    gather_max_phi_kernel<<<ceil_div(n, 128), 128, 0, s>>>((const char*)d_stats, sizeof(mavd_frame_stats), n, d_out);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Residual angle phi + the two masks + the integer reductions behind FrameResult.
//
// MODE 0  float32 flow + IMU derotation, all arithmetic in float64 (frames with imu.derotate != 0)
// MODE 1  float32 flow passed through (frame_index < 1): NumPy keeps every temporary in float32
// MODE 2  float64 flow given by the caller, no derotation (FocusOfExpansion.get_phi on any array)
//
// Derotation uses host-built tables xn[x] = -(x/w - 0.5)*2, yn[y] = -(y/h - 0.5)*2 (IEEE doubles, the
// same values NumPy computes), so the per-pixel float64 work has no division.
//
// FAST (MODE 0/2, phi not requested): the masks are decided from a float32 estimate of phi
// (atan2 of cross and dot product, well conditioned at every angle) whenever the estimate is further
// from every threshold than a conservative error bound; only pixels inside the guard bands (and any
// non-finite or degenerate input) take the exact float64 path below.  Masks and counts stay
// bit-exact; max_phi is not evaluated on this path (reported as -1).
// ------------------------------------------------------------------------------------------------
struct ResidualPrm {
    double dyn_offset, dyn_base, dyn_gain, dyn_min_mag, fixed_min_mag, fixed_angle;
};

struct ResidualArgs {
    const void* flow;
    const mavd_imu* imu;     // NULL for flow kinds that ignore the IMU
    const double* foe;
    const double* xn;
    const double* yn;
    int w, h;
    ResidualPrm prm;
    const uint8_t* sky; int64_t sky_stride;
    const uint8_t* seg; int64_t seg_stride;
    const int* seg_max;
    const float2* gt_flow;   // nullable: ground-truth flow, summed (derotated) over segmentation > 127
    void* phi_out;
    uint8_t* total_out;
    uint8_t* fixed_out;
    char* stats_base; size_t stats_stride;
    unsigned row_magic;      // 0, or M with i0 / w == __umulhi(i0, M) for every pixel index of a frame (host-checked)
    int* unit_marks; int* unit_list; int* unit_count; int n_units;   // nullable: list of occupied units of the fixed mask (see ccl_*)
};

__device__ __forceinline__ unsigned long long dmax_key(double v) { return (unsigned long long)__double_as_longlong(v); }

// max over a uint8 image, 16 bytes per load where the alignment allows
__global__ void __launch_bounds__(256) seg_max_kernel(const uint8_t* __restrict__ seg, int64_t seg_stride, int64_t npx,
                                                     int* __restrict__ seg_max) {
    pdl_entry();
    const int f = blockIdx.y;
    const uint8_t* p = seg + (size_t)f * seg_stride;
    unsigned mx4 = 0;
    int mx = 0;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
        const int64_t n16 = npx >> 4;
        const uint4* p16 = reinterpret_cast<const uint4*>(p);
        for (int64_t i = tid; i < n16; i += nthr) {
            const uint4 v = __ldg(p16 + i);
            mx4 = __vmaxu4(mx4, __vmaxu4(__vmaxu4(v.x, v.y), __vmaxu4(v.z, v.w)));
        }
        for (int64_t i = (n16 << 4) + tid; i < npx; i += nthr) mx = max(mx, (int)p[i]);
    } else {
        for (int64_t i = tid; i < npx; i += nthr) mx = max(mx, (int)p[i]);
    }
    mx = max(mx, (int)max(max(mx4 & 255u, (mx4 >> 8) & 255u), max((mx4 >> 16) & 255u, mx4 >> 24)));
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(seg_max + f, mx);
}

struct DerotRow {   // per-frame, per-row constants of detector.py:93-101 (NumPy operation order)
    double o0, o1, o2, s0, s1;
    int on;
};

__device__ __forceinline__ void derot_tab(const DerotRow& d, double xn, double yn, double& r0, double& r1) {
    double t = __dmul_rn(__dmul_rn(d.o0, xn), yn);
    t = __dsub_rn(t, __dmul_rn(d.o1, __dmul_rn(xn, xn)));
    t = __dsub_rn(t, d.o1);
    t = __dadd_rn(t, __dmul_rn(d.o2, yn));
    r0 = __dmul_rn(t, d.s0);
    double u = __dmul_rn(-d.o2, xn);
    u = __dadd_rn(u, d.o0);
    u = __dadd_rn(u, __dmul_rn(d.o0, __dmul_rn(yn, yn)));
    u = __dsub_rn(u, __dmul_rn(__dmul_rn(d.o1, xn), yn));
    r1 = __dmul_rn(u, d.s1);
}

// exact float64 evaluation of focus_of_expansion.py:165-178 and processor.py:333-341 for one pixel
__device__ __forceinline__ void pixel_exact_f64(double fdx, double fdy, int x, int y, double foex, double foey,
                                                const ResidualPrm& prm, bool not_sky, bool& m_total, bool& m_fixed,
                                                double& phi) {
    const double d2x = __dsub_rn((double)x, foex), d2y = __dsub_rn((double)y, foey);
    const double a = __dsqrt_rn(__dadd_rn(__dmul_rn(fdx, fdx), __dmul_rn(fdy, fdy)));
    const double b = __dsqrt_rn(__dadd_rn(__dmul_rn(d2x, d2x), __dmul_rn(d2y, d2y)));
    const double ab = __dmul_rn(a, b);
    const double norm = (ab != ab) ? ab : fmax(1e-6, ab);
    double c = __ddiv_rn(__dadd_rn(__dmul_rn(fdx, d2x), __dmul_rn(fdy, d2y)), norm);
    if (c == c) c = fmin(fmax(c, -1.0), 1.0);
    double ang = acos(c);
    if (ang != ang) ang = 0.0;
    phi = __dmul_rn(ang, 180.0 / 3.141592653589793238462643383279502884);
    const double t = __dadd_rn(prm.dyn_base, __ddiv_rn(prm.dyn_gain, a));
    const bool amax = phi > __dadd_rn(prm.dyn_offset, t);
    const bool amin = phi < __dsub_rn(prm.dyn_offset, t);
    m_total = (a > prm.dyn_min_mag) && not_sky && (amin || amax);
    m_fixed = (((a > prm.fixed_min_mag) && not_sky) ? phi : 0.0) > prm.fixed_angle;
}

__device__ __forceinline__ void pixel_exact_f32(float fx, float fy, int x, int y, double foex, double foey,
                                                const ResidualPrm& prm, bool not_sky, bool& m_total, bool& m_fixed,
                                                float& phi) {
    // the flow stays float32 and so does every NumPy temporary (diff2 = zeros_like(flow))
    const float d2x = (float)__dsub_rn((double)x, foex), d2y = (float)__dsub_rn((double)y, foey);
    const float a = __fsqrt_rn(__fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy)));
    const float b = __fsqrt_rn(__fadd_rn(__fmul_rn(d2x, d2x), __fmul_rn(d2y, d2y)));
    const float ab = __fmul_rn(a, b);
    const float norm = (ab != ab) ? ab : fmaxf(1e-6f, ab);
    float c = __fdiv_rn(__fadd_rn(__fmul_rn(fx, d2x), __fmul_rn(fy, d2y)), norm);
    if (c == c) c = fminf(fmaxf(c, -1.f), 1.f);
    float ang = (float)acos((double)c);
    if (ang != ang) ang = 0.f;
    phi = __fmul_rn(ang, 180.0f / 3.141592653589793238462643383279502884f);
    const float t = __fadd_rn((float)prm.dyn_base, __fdiv_rn((float)prm.dyn_gain, a));
    const bool amax = phi > __fadd_rn((float)prm.dyn_offset, t);
    const bool amin = phi < __fsub_rn((float)prm.dyn_offset, t);
    m_total = (a > (float)prm.dyn_min_mag) && not_sky && (amin || amax);
    m_fixed = (((a > (float)prm.fixed_min_mag) && not_sky) ? phi : 0.f) > (float)prm.fixed_angle;
}

// float32 pre-decision, branch-free and without an inverse trigonometric function.  Returns false when the pixel
// must take the exact path.
//   phi > T  <=>  sin(phi - T) > 0  <=>  crs * cos T - dot * sin T > 0      (phi, T in [0, 180) degrees)
// with dot = f . d and crs = |f x d| (so that |f||d| sin(phi - T) is the tested quantity).  Error budget, relative
// to |f||d|: inputs rounded once to float32 (6e-8 each), dot / crs with FMAs (< 4e-7), __sincosf (< 5e-7), the
// dynamic threshold through rsqrtf (2 ulp) -> under 3e-6 in total.  A pixel is decided here only when
// |sin(phi - T)| > 3.6e-5 (2e-3 degrees, plus 1e-5 relative on the dynamic threshold) and the squared magnitude is
// further than 1e-5 relative from both magnitude gates; everything else, and any non-finite, huge or degenerate
// input, takes the float64 path.  The reference's own evaluation (float64 arccos) is within 1e-12 of the exact angle
// at every threshold in range, so both sides agree on all pixels decided here.
struct FastPrm {
    float dyn_c0;                     // dyn_offset + dyn_base, degrees
    float dyn_gain;                   // degrees x pixels
    float dyn_mm2, fix_mm2;           // squared magnitude gates
    float dyn_mm2_guard, fix_mm2_guard;
    float fix_cos, fix_sin;           // of the fixed angle threshold
};

__device__ __forceinline__ bool pixel_fast(float fx, float fy, float dx, float dy, const FastPrm& p, bool& m_total,
                                           bool& m_fixed) {
    const float a2 = fmaf(fx, fx, fy * fy), b2 = fmaf(dx, dx, dy * dy);
    const float ab2 = a2 * b2;
    const bool gt_dyn = a2 > p.dyn_mm2, gt_fix = a2 > p.fix_mm2;
    bool undecided = !(a2 < 1e15f) | !(b2 < 1e15f);                         // NaN / inf / huge
    undecided |= (fabsf(a2 - p.dyn_mm2) <= p.dyn_mm2_guard) | (fabsf(a2 - p.fix_mm2) <= p.fix_mm2_guard);
    const float dot = fmaf(fx, dx, fy * dy), crs = fabsf(fmaf(fx, dy, -(fy * dx)));
    const float sf = crs * p.fix_cos - dot * p.fix_sin;
    const float thr = fmaf(p.dyn_gain, rsqrtf(a2), p.dyn_c0);               // degrees; inf when a2 == 0 (then !gt_dyn)
    const float tr = thr * 0.017453292519943295f;
    float sn, cs;
    __sincosf(tr, &sn, &cs);
    const float sd = crs * cs - dot * sn;
    const float mf = 3.6e-5f, md = 3.6e-5f + 1e-5f * tr;
    undecided |= (gt_dyn | gt_fix) & (ab2 < 1e-8f);                         // |f||d| near the 1e-6 clamp of the norm
    undecided |= gt_fix & (sf * sf <= (mf * mf) * ab2);
    undecided |= gt_dyn & ((sd * sd <= (md * md) * ab2) | !(thr < 170.f));
    m_fixed = gt_fix & (sf > 0.f);
    m_total = gt_dyn & (sd > 0.f);      // amin is impossible: the host enables FAST only when offset - base < 0
    return !undecided;
}

constexpr int RES_ITEMS = 4;     // pixel groups per thread

// MINB: CTAs per SM the register allocation aims at.  4 (64 registers) is the best for frames that derotate; a batch
// whose derotating frames all have a zero rotation (the host sees the imu array) never enters the float64 derotation and
// runs 9 % faster at 5 (48 registers).  Only the register budget differs: the kernel still decides per frame from the
// device copy of the imu data, so a wrong hint costs time, never correctness.
template <int MODE, bool FAST, int VEC, int MINB = 4>
__global__ void __launch_bounds__(256, MINB) residual_kernel(const ResidualArgs A, const FastPrm fp) {
    pdl_entry();
    const int f = blockIdx.y;
    DerotRow dr;
    dr.on = 0;
    if (MODE != 2) {
        mavd_imu im;
        im.derotate = 0;
        if (A.imu) im = A.imu[f];
        // every mode is launched over the whole batch; each handles only its own frames
        if ((im.derotate != 0) != (MODE == 0)) return;
        if (MODE == 0) {
            // the five float64 divisions are done once per block (one thread each), not once per thread: they were
            // 150 of the ~2200 instructions a thread executes
            __shared__ double s_dr[5];
            if (threadIdx.x < 3) s_dr[threadIdx.x] = __ddiv_rn(im.ang[threadIdx.x], im.dt);
            else if (threadIdx.x == 3) s_dr[3] = __ddiv_rn(__dmul_rn((double)A.w, im.dt), 2.0);
            else if (threadIdx.x == 4) s_dr[4] = __ddiv_rn(__dmul_rn((double)A.h, im.dt), 2.0);
            __syncthreads();
            dr.o0 = s_dr[0]; dr.o1 = s_dr[1]; dr.o2 = s_dr[2]; dr.s0 = s_dr[3]; dr.s1 = s_dr[4];
            // omega == 0 and finite scales: the derotation field is exactly (+-)0 and flow - 0 == flow
            dr.on = !(dr.o0 == 0.0 && dr.o1 == 0.0 && dr.o2 == 0.0 && fabs(dr.s0) < 1e300 && fabs(dr.s1) < 1e300);
        }
    }
    const int w = A.w, h = A.h;
    const int npx = w * h;
    const int ngrp = npx / VEC;                 // VEC == 4 only when w % 4 == 0
    const double foex = A.foe[2 * f], foey = A.foe[2 * f + 1];
    const size_t fbase = (size_t)f * npx;
    const uint8_t* sky = A.sky ? A.sky + (size_t)f * A.sky_stride : nullptr;
    const uint8_t* seg = A.seg ? A.seg + (size_t)f * A.seg_stride : nullptr;
    const bool want_stats = A.stats_base != nullptr;
    // g > 0.1 * max  <=>  g >= seg_min (g integer): the largest integer not above the float64 threshold, plus one
    int seg_min = 0;
    if (seg && want_stats) {
        const double thr = 0.1 * (double)A.seg_max[f];
        seg_min = (int)floor(thr) + 1;
    }

    int c_tot = 0, c_fix = 0, c_pos = 0, c_tpt = 0, c_fpt = 0, c_tpf = 0, c_fpf = 0, n_px = 0;
    int bx0 = 0x7fffffff, by0 = 0x7fffffff, bx1 = -1, by1 = -1;
    double sfx = 0.0, sfy = 0.0, gfx = 0.0, gfy = 0.0, maxphi = 0.0;

#pragma unroll 1
    for (int it = 0; it < RES_ITEMS; ++it) {
        const int q = (blockIdx.x * RES_ITEMS + it) * 256 + threadIdx.x;
        if (q >= ngrp) break;
        const int i0 = q * VEC;
        const int y = A.row_magic ? (int)__umulhi((unsigned)i0, A.row_magic) : i0 / w, x0 = i0 - y * w;
        // ---- loads ----
        double vx[VEC], vy[VEC];
        float vfx[VEC], vfy[VEC];
        if (MODE == 2) {
            const double2* fl = reinterpret_cast<const double2*>(A.flow) + fbase + i0;
#pragma unroll
            for (int k = 0; k < VEC; ++k) { const double2 v = fl[k]; vx[k] = v.x; vy[k] = v.y; }
        } else if (VEC == 4) {
            const float4* fl = reinterpret_cast<const float4*>(reinterpret_cast<const float2*>(A.flow) + fbase + i0);
            const float4 u0 = __ldg(fl), u1 = __ldg(fl + 1);
            vfx[0] = u0.x; vfy[0] = u0.y; vfx[1] = u0.z; vfy[1] = u0.w;
            vfx[2] = u1.x; vfy[2] = u1.y; vfx[3] = u1.z; vfy[3] = u1.w;
        } else {
            const float2 v = reinterpret_cast<const float2*>(A.flow)[fbase + i0];
            vfx[0] = v.x; vfy[0] = v.y;
        }
        unsigned skyw = 0, segw = 0;
        if (VEC == 4) {
            if (sky) skyw = __ldg(reinterpret_cast<const unsigned*>(sky + i0));
            if (seg) segw = __ldg(reinterpret_cast<const unsigned*>(seg + i0));
        } else {
            if (sky) skyw = sky[i0];
            if (seg) segw = seg[i0];
        }
        double yn = 0.0;
        if (MODE == 0 && dr.on) yn = __ldg(A.yn + y);
        // FAST: FoE ray components in float32 (x0 + k in float adds one rounding, 6e-8 relative: inside the budget)
        const float dyf = (float)((double)y - foey), dxf0 = (float)((double)x0 - foex);
        unsigned totw = 0, fixw = 0;
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            const int x = x0 + k;
            const bool not_sky = ((skyw >> (8 * k)) & 255u) == 0;
            bool mt = false, mf = false;
            if (MODE == 1) {
                float phi;
                pixel_exact_f32(vfx[k], vfy[k], x, y, foex, foey, A.prm, not_sky, mt, mf, phi);
                maxphi = fmax(maxphi, (double)phi);
                if (A.phi_out) reinterpret_cast<float*>(reinterpret_cast<double*>(A.phi_out) + fbase)[i0 + k] = phi;
            } else {
                double fdx = 0.0, fdy = 0.0;
                bool decided = false;
                if (FAST && MODE == 0 && !dr.on) {
                    // no derotation: the float64 flow IS the float32 input, doubles are needed on the exact path only
                    decided = !not_sky;                // both masks are multiplied by ~sky
                    if (!decided) decided = pixel_fast(vfx[k], vfy[k], dxf0 + (float)k, dyf, fp, mt, mf);
                    if (!decided) { fdx = (double)vfx[k]; fdy = (double)vfy[k]; }
                } else {
                    if (MODE == 0) {
                        fdx = vfx[k]; fdy = vfy[k];
                        if (dr.on) {
                            double r0, r1;
                            derot_tab(dr, __ldg(A.xn + x), yn, r0, r1);
                            fdx = __dsub_rn(fdx, r0);
                            fdy = __dsub_rn(fdy, r1);
                        }
                    } else {
                        fdx = vx[k]; fdy = vy[k];
                    }
                    vx[k] = fdx; vy[k] = fdy;          // kept for the flow sum over the segmentation below
                    if (FAST) {
                        if (!not_sky) decided = true;
                        else decided = pixel_fast((float)fdx, (float)fdy, dxf0 + (float)k, dyf, fp, mt, mf);
                    }
                }
                if (!decided) {
                    double phi;
                    pixel_exact_f64(fdx, fdy, x, y, foex, foey, A.prm, not_sky, mt, mf, phi);
                    if (!FAST) {
                        maxphi = fmax(maxphi, phi);
                        if (A.phi_out) reinterpret_cast<double*>(A.phi_out)[fbase + i0 + k] = phi;
                    }
                }
            }
            totw |= (mt ? 1u : 0u) << (8 * k);
            fixw |= (mf ? 1u : 0u) << (8 * k);
        }
        if (A.unit_marks && fixw) {
            // append the 128-pixel unit to the list the labelling passes walk (once per unit: the mark decides)
            const int e = f * A.n_units + (i0 >> 7);
            if (*reinterpret_cast<volatile int*>(A.unit_marks + e) == 0 && atomicExch(A.unit_marks + e, 1) == 0)
                A.unit_list[atomicAdd(A.unit_count, 1)] = e;
        }
        n_px += VEC;
        if (want_stats && (totw | fixw | segw)) {
            // counts on whole words: mask bytes are 0/1, segmentation bytes are tested with per-byte compares
            // (words with empty masks and an empty segmentation, almost all of them, add nothing but negatives,
            // which are counted as pixels seen minus positives at the end)
            c_tot += __popc(totw); c_fix += __popc(fixw);
            if (seg) {
                const unsigned live = VEC == 4 ? 0xffffffffu : 0xffu;
                const unsigned hi = segw & 0x80808080u & live;                        // g > 127
                const unsigned nz = __vcmpne4(segw, 0u) & 0x01010101u & live;          // g >= 1
                const unsigned n255 = __vcmpne4(segw, 0xffffffffu) & 0x01010101u & live;   // g <= 254
                c_pos += __popc(hi);
                c_tpt += __popc(totw & nz); c_fpt += __popc(totw & n255);
                c_tpf += __popc(fixw & nz); c_fpf += __popc(fixw & n255);
                const unsigned smin = (unsigned)min(seg_min, 256);
                const unsigned ge = smin > 255u ? 0u : (__vcmpgeu4(segw, smin * 0x01010101u) & live);
                if (ge) {
                    bx0 = min(bx0, x0 + ((__ffs(ge) - 1) >> 3)); bx1 = max(bx1, x0 + ((31 - __clz(ge)) >> 3));
                    by0 = min(by0, y); by1 = max(by1, y);
                }
                if (hi) {
#pragma unroll
                    for (int k = 0; k < VEC; ++k)
                        if ((hi >> (8 * k)) & 0x80u) {
                            if (MODE == 1 || (FAST && MODE == 0 && !dr.on)) { sfx += (double)vfx[k]; sfy += (double)vfy[k]; }
                            else { sfx += vx[k]; sfy += vy[k]; }
                            if (MODE != 2 && A.gt_flow) {
                                // Detector.derotate on the ground-truth flow (processor.py:309-310), only where it is
                                // summed (processor.py:344): a few hundred pixels per frame
                                const float2 g = __ldg(A.gt_flow + fbase + i0 + k);
                                double g0 = (double)g.x, g1 = (double)g.y;
                                if (MODE == 0 && dr.on) {
                                    double r0, r1;
                                    derot_tab(dr, __ldg(A.xn + x0 + k), yn, r0, r1);
                                    g0 = __dsub_rn(g0, r0);
                                    g1 = __dsub_rn(g1, r1);
                                }
                                gfx += g0; gfy += g1;
                            }
                        }
                }
            }
        }
        if (VEC == 4) {
            if (A.total_out) *reinterpret_cast<unsigned*>(A.total_out + fbase + i0) = totw;
            if (A.fixed_out) *reinterpret_cast<unsigned*>(A.fixed_out + fbase + i0) = fixw;
        } else {
            if (A.total_out) A.total_out[fbase + i0] = (uint8_t)totw;
            if (A.fixed_out) A.fixed_out[fbase + i0] = (uint8_t)fixw;
        }
    }
    if (!want_stats) return;

    // ---- block reduction: warp redux -> shared atomics -> one set of global atomics per block ----
    __shared__ int s_cnt[8];
    __shared__ int s_bb[4];
    __shared__ double s_sum[4];
    __shared__ unsigned long long s_max;
    if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 8) {
        s_bb[0] = s_bb[1] = 0x7fffffff; s_bb[2] = s_bb[3] = -1;
        s_sum[0] = s_sum[1] = s_sum[2] = s_sum[3] = 0.0; s_max = 0ull;
    }
    __syncthreads();
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    c_tot = __reduce_add_sync(FULL, c_tot); c_fix = __reduce_add_sync(FULL, c_fix);
    if (lane == 0) { if (c_tot) atomicAdd(&s_cnt[0], c_tot); if (c_fix) atomicAdd(&s_cnt[1], c_fix); }
    if (!FAST) {
        unsigned long long mk = dmax_key(maxphi);
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const unsigned long long t = __shfl_xor_sync(FULL, mk, s);
            mk = t > mk ? t : mk;
        }
        if (lane == 0 && mk) atomicMax(&s_max, mk);
    }
    if (seg) {
        int c_neg = n_px - c_pos;      // 255 - g > 127 <=> not (g > 127)
        c_pos = __reduce_add_sync(FULL, c_pos); c_neg = __reduce_add_sync(FULL, c_neg);
        c_tpt = __reduce_add_sync(FULL, c_tpt); c_fpt = __reduce_add_sync(FULL, c_fpt);
        c_tpf = __reduce_add_sync(FULL, c_tpf); c_fpf = __reduce_add_sync(FULL, c_fpf);
        bx0 = __reduce_min_sync(FULL, bx0); by0 = __reduce_min_sync(FULL, by0);
        bx1 = __reduce_max_sync(FULL, bx1); by1 = __reduce_max_sync(FULL, by1);
        const bool any_sum = __any_sync(FULL, sfx != 0.0 || sfy != 0.0 || gfx != 0.0 || gfy != 0.0);
        if (any_sum) {
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) {
                sfx += __shfl_xor_sync(FULL, sfx, s);
                sfy += __shfl_xor_sync(FULL, sfy, s);
                gfx += __shfl_xor_sync(FULL, gfx, s);
                gfy += __shfl_xor_sync(FULL, gfy, s);
            }
        }
        if (lane == 0) {
            if (c_pos) atomicAdd(&s_cnt[2], c_pos);
            if (c_neg) atomicAdd(&s_cnt[3], c_neg);
            if (c_tpt) atomicAdd(&s_cnt[4], c_tpt);
            if (c_fpt) atomicAdd(&s_cnt[5], c_fpt);
            if (c_tpf) atomicAdd(&s_cnt[6], c_tpf);
            if (c_fpf) atomicAdd(&s_cnt[7], c_fpf);
            if (bx1 >= 0) { atomicMin(&s_bb[0], bx0); atomicMin(&s_bb[1], by0); atomicMax(&s_bb[2], bx1); atomicMax(&s_bb[3], by1); }
            if (any_sum) {
                atomicAdd(&s_sum[0], sfx); atomicAdd(&s_sum[1], sfy);
                if (gfx != 0.0) atomicAdd(&s_sum[2], gfx);
                if (gfy != 0.0) atomicAdd(&s_sum[3], gfy);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mavd_frame_stats* st = reinterpret_cast<mavd_frame_stats*>(A.stats_base + (size_t)f * A.stats_stride);
        typedef unsigned long long ull;
        if (s_cnt[0]) atomicAdd((ull*)&st->n_total, (ull)s_cnt[0]);
        if (s_cnt[1]) atomicAdd((ull*)&st->n_fixed, (ull)s_cnt[1]);
        if (!FAST && s_max) atomicMax((ull*)&st->max_phi, s_max);
        if (seg) {
            if (s_cnt[2]) atomicAdd((ull*)&st->positives, (ull)s_cnt[2]);
            if (s_cnt[3]) atomicAdd((ull*)&st->negatives, (ull)s_cnt[3]);
            if (s_cnt[4]) atomicAdd((ull*)&st->tp_total, (ull)s_cnt[4]);
            if (s_cnt[5]) atomicAdd((ull*)&st->fp_total, (ull)s_cnt[5]);
            if (s_cnt[6]) atomicAdd((ull*)&st->tp_fixed, (ull)s_cnt[6]);
            if (s_cnt[7]) atomicAdd((ull*)&st->fp_fixed, (ull)s_cnt[7]);
            if (s_bb[2] >= 0) {
                // seg_bbox was initialised to {INT_MAX, INT_MAX, -1, -1} by stats_init_kernel
                atomicMin(&st->seg_bbox[0], s_bb[0]); atomicMin(&st->seg_bbox[1], s_bb[1]);
                atomicMax(&st->seg_bbox[2], s_bb[2]); atomicMax(&st->seg_bbox[3], s_bb[3]);
            }
            if (s_sum[0] != 0.0) atomicAdd(&st->seg_flow_sum[0], s_sum[0]);
            if (s_sum[1] != 0.0) atomicAdd(&st->seg_flow_sum[1], s_sum[1]);
            if (s_sum[2] != 0.0) atomicAdd(&st->gt_flow_sum[0], s_sum[2]);
            if (s_sum[3] != 0.0) atomicAdd(&st->gt_flow_sum[1], s_sum[3]);
        }
    }
}

__global__ void stats_init_kernel(char* stats_base, size_t stats_stride, int n, int* seg_max) {
    pdl_entry();
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    mavd_frame_stats* st = reinterpret_cast<mavd_frame_stats*>(stats_base + (size_t)f * stats_stride);
    mavd_frame_stats z;
    memset(&z, 0, sizeof(z));
    z.seg_bbox[0] = z.seg_bbox[1] = 0x7fffffff;
    z.seg_bbox[2] = z.seg_bbox[3] = -1;
    *st = z;
    if (seg_max) seg_max[f] = 0;
}

// no_max_phi: the FAST path ran (for the frames with imu.derotate != 0, or for all frames when imu is NULL)
__global__ void stats_final_kernel(char* stats_base, size_t stats_stride, int n, int no_max_phi, const mavd_imu* imu) {
    pdl_entry();
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    mavd_frame_stats* st = reinterpret_cast<mavd_frame_stats*>(stats_base + (size_t)f * stats_stride);
    if (st->seg_bbox[2] < 0) st->seg_bbox[0] = st->seg_bbox[1] = st->seg_bbox[2] = st->seg_bbox[3] = -1;
    if (no_max_phi && (imu == nullptr || imu[f].derotate != 0)) st->max_phi = -1.0;
}

template <int MODE, bool FAST>
static int launch_residual(const ResidualArgs& A, const FastPrm& fp, int n, bool vec4, cudaStream_t s, bool pdl,
                           bool no_rotation = false) {
    const int npx = A.w * A.h;
    if (vec4 && no_rotation && MODE == 0 && FAST) {
        dim3 g(ceil_div(npx / 4, 256 * RES_ITEMS), n);
        MAVD_CUDA(launch_chained(pdl, residual_kernel<MODE, FAST, 4, (MODE == 0 && FAST) ? 5 : 4>, g, 256, 0, s, A, fp));
    } else if (vec4) {
        dim3 g(ceil_div(npx / 4, 256 * RES_ITEMS), n);
        MAVD_CUDA(launch_chained(pdl, residual_kernel<MODE, FAST, 4>, g, 256, 0, s, A, fp));
    } else {
        dim3 g(ceil_div(npx, 256 * RES_ITEMS), n);
        MAVD_CUDA(launch_chained(pdl, residual_kernel<MODE, FAST, 1>, g, 256, 0, s, A, fp));
    }
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// flow_kind: 0 = float32 flow with the per-frame imu deciding between MODE 0 and MODE 1,
//            1 = float32 flow, no derotation for any frame (MODE 1), 2 = float64 flow, no derotation (MODE 2)
// run_f64:   0 = no frame derotates, 1 = some do, 2 = some do and none of them by a non-zero rotation (the register
//            budget hint of residual_kernel's MINB)
// What the residual kernel needs besides the flow and the FoE: zeroed statistics and the per-frame maximum of the
// segmentation (get_simple_bounding_box's threshold).  Independent of both, so the batch call (api.cu: detect_run) runs
// it on the side stream (lane 1) while the FoE estimation, 64 CTAs, has the GPU almost to itself.
int residual_prepare(mavd_handle H, int n, const uint8_t* d_seg, int64_t seg_stride, mavd_frame_stats* d_stats,
                     size_t stats_stride, cudaStream_t s, int lane) {
    if (!d_stats) return MAVD_OK;
    ProfScope ps(&H->prof, MAVD_PROF_RESIDUAL, s);
    int* seg_max = reinterpret_cast<int*>(H->d_scan);  // scratch: n ints
    MAVD_CUDA(launch_chained(pdl_next(H, lane), stats_init_kernel, ceil_div(n, 128), 128, 0, s, (char*)d_stats, stats_stride, n,
                             d_seg ? seg_max : nullptr));
    MAVD_LAUNCHED();
    if (d_seg) {
        dim3 g(32, n);
        MAVD_CUDA(launch_chained(pdl_next(H, lane), seg_max_kernel, g, 256, 0, s, d_seg, seg_stride,
                                 (int64_t)H->cfg.width * H->cfg.height, seg_max));
        MAVD_LAUNCHED();
    }
    return MAVD_OK;
}

int residual_run(mavd_handle H, const void* d_flow, int flow_kind, int n, const mavd_imu* d_imu,
                 const mavd_detect_params& p, const double* d_foe, const uint8_t* d_sky, int64_t sky_stride,
                 const uint8_t* d_seg, int64_t seg_stride, void* d_phi, uint8_t* d_total, uint8_t* d_fixed,
                 mavd_frame_stats* d_stats, size_t stats_stride, int run_f64, int run_f32, cudaStream_t s,
                 bool list_fixed_units, const float* d_gt_flow, bool prepared) {
    if (!prepared) TRY_RC(residual_prepare(H, n, d_seg, seg_stride, d_stats, stats_stride, s, 0));
    ProfScope ps(&H->prof, MAVD_PROF_RESIDUAL, s);
    const int w = H->cfg.width, h = H->cfg.height;
    const int64_t npx = (int64_t)w * h;
    int* seg_max = reinterpret_cast<int*>(H->d_scan);  // scratch: n ints
    // FAST needs: phi not requested, and the parameter ranges its guard bands were derived for
    const bool fast = !H->force_exact_residual && d_phi == nullptr && p.fixed_angle >= 0.0 && p.dyn_gain >= 0.0 &&
                      p.dyn_offset - p.dyn_base < -1e-2 && p.dyn_min_mag >= 0.0 && p.fixed_min_mag >= 0.0 &&
                      p.fixed_angle <= 170.0 && p.dyn_offset + p.dyn_base < 160.0 && p.dyn_gain < 1e6 &&
                      p.dyn_min_mag < 1e3 && p.fixed_min_mag < 1e3;
    ResidualArgs A;
    A.flow = d_flow; A.imu = flow_kind == 0 ? d_imu : nullptr; A.foe = d_foe; A.xn = H->d_xn; A.yn = H->d_yn; A.w = w; A.h = h;
    A.prm = ResidualPrm{p.dyn_offset, p.dyn_base, p.dyn_gain, p.dyn_min_mag, p.fixed_min_mag, p.fixed_angle};
    A.sky = d_sky; A.sky_stride = sky_stride; A.seg = d_seg; A.seg_stride = seg_stride; A.seg_max = seg_max;
    A.gt_flow = (d_seg && d_stats) ? reinterpret_cast<const float2*>(d_gt_flow) : nullptr;
    A.phi_out = d_phi; A.total_out = d_total; A.fixed_out = d_fixed;
    A.stats_base = (char*)d_stats; A.stats_stride = stats_stride;
    // i / w by multiplication: M = floor(2^32 / w) + 1 is exact for i * (M * w - 2^32) < 2^32
    {
        const unsigned long long M = (1ull << 32) / (unsigned)w + 1, err = M * (unsigned)w - (1ull << 32);
        A.row_magic = (M < (1ull << 32) && (unsigned long long)npx * err < (1ull << 32)) ? (unsigned)M : 0u;
    }
    const bool listing = list_fixed_units && d_fixed != nullptr;
    A.unit_marks = listing ? ccl_unit_marks(H) : nullptr; A.unit_list = listing ? ccl_unit_list(H) : nullptr;
    A.unit_count = listing ? ccl_unit_count(H) : nullptr; A.n_units = ccl_n_units(H);
    auto gate_guard = [](double t) { const double g = 1e-5 * (t > 1.0 ? t : 1.0); return (float)(2.0 * t * g + g * g); };
    const double fixed_rad = p.fixed_angle * (3.14159265358979323846 / 180.0);
    const FastPrm fp{(float)(p.dyn_offset + p.dyn_base), (float)p.dyn_gain,
                     (float)(p.dyn_min_mag * p.dyn_min_mag), (float)(p.fixed_min_mag * p.fixed_min_mag),
                     gate_guard(p.dyn_min_mag), gate_guard(p.fixed_min_mag), (float)cos(fixed_rad), (float)sin(fixed_rad)};
    auto al = [](const void* q, uintptr_t a) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & (a - 1)) == 0; };
    const bool vec4 = (w % 4 == 0) && al(d_flow, 16) && al(d_sky, 4) && al(d_seg, 4) && al(d_total, 4) && al(d_fixed, 4) &&
                      (sky_stride % 4 == 0) && (seg_stride % 4 == 0);
    bool used_fast = false;
    if (flow_kind == 2) {
        if (fast) { used_fast = true; TRY_RC(launch_residual<2, true>(A, fp, n, vec4, s, pdl_next(H))); }
        else      TRY_RC(launch_residual<2, false>(A, fp, n, vec4, s, pdl_next(H)));
    } else {
        if (flow_kind == 0 && run_f64) {
            if (fast) { used_fast = true; TRY_RC(launch_residual<0, true>(A, fp, n, vec4, s, pdl_next(H), run_f64 == 2)); }
            else      TRY_RC(launch_residual<0, false>(A, fp, n, vec4, s, pdl_next(H)));
        }
        if (flow_kind == 1 || run_f32) TRY_RC(launch_residual<1, false>(A, fp, n, vec4, s, pdl_next(H)));
    }
    if (d_stats) {
        MAVD_CUDA(launch_chained(pdl_next(H), stats_final_kernel, ceil_div(n, 128), 128, 0, s, (char*)d_stats, stats_stride, n,
                                 used_fast ? 1 : 0, A.imu));
        MAVD_LAUNCHED();
    }
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Stand-alone im_helpers seams (im_helpers.py:150-159, 55-84, 244-252) for callers that use them outside
// the fused residual kernel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) magnitude_kernel(const void* __restrict__ flow, int is_f64, int64_t n,
                                                       void* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (is_f64) {
        const double2 v = reinterpret_cast<const double2*>(flow)[i];
        reinterpret_cast<double*>(out)[i] = __dsqrt_rn(__dadd_rn(__dmul_rn(v.x, v.x), __dmul_rn(v.y, v.y)));
    } else {
        const float2 v = reinterpret_cast<const float2*>(flow)[i];
        reinterpret_cast<float*>(out)[i] = __fsqrt_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)));
    }
}

int magnitude_run(const void* d_flow, int is_f64, int64_t n, void* d_out, cudaStream_t s) {
    magnitude_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_flow, is_f64, n, d_out);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

__global__ void bbox_init_kernel(int32_t* out5) {
    out5[0] = out5[1] = 0x7fffffff;
    out5[2] = out5[3] = -1;
    out5[4] = 0;
}

// out5 = {x0, y0, x1, y1, max}; element e of the (H, W, C) image belongs to column (e % (W*C)) / C
__global__ void __launch_bounds__(256) bbox_kernel(const uint8_t* __restrict__ img, int w, int h, int c,
                                                  int32_t* __restrict__ out5) {
    const double thr = 0.1 * (double)out5[4];
    const int64_t n = (int64_t)w * h * c, rowlen = (int64_t)w * c;
    int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        if ((double)img[e] > thr) {
            const int y = (int)(e / rowlen), x = (int)((e - (int64_t)y * rowlen) / c);
            x0 = min(x0, x); x1 = max(x1, x); y0 = min(y0, y); y1 = max(y1, y);
        }
    }
    x0 = __reduce_min_sync(0xffffffffu, x0); y0 = __reduce_min_sync(0xffffffffu, y0);
    x1 = __reduce_max_sync(0xffffffffu, x1); y1 = __reduce_max_sync(0xffffffffu, y1);
    if ((threadIdx.x & 31) == 0 && x1 >= 0) {
        atomicMin(out5 + 0, x0); atomicMin(out5 + 1, y0); atomicMax(out5 + 2, x1); atomicMax(out5 + 3, y1);
    }
}

__global__ void bbox_final_kernel(int32_t* out5) {
    if (out5[2] < 0) out5[0] = out5[1] = out5[2] = out5[3] = -1;
}

int simple_bbox_run(const uint8_t* d_img, int w, int h, int c, int32_t* d_out5, cudaStream_t s) {
    const int64_t n = (int64_t)w * h * c;
    bbox_init_kernel<<<1, 1, 0, s>>>(d_out5);
    MAVD_LAUNCHED();
    seg_max_kernel<<<dim3(148, 1), 256, 0, s>>>(d_img, 0, n, d_out5 + 4);
    MAVD_LAUNCHED();
    bbox_kernel<<<148 * 4, 256, 0, s>>>(d_img, w, h, c, d_out5);
    MAVD_LAUNCHED();
    bbox_final_kernel<<<1, 1, 0, s>>>(d_out5);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// counts4 = {sum(gt > 127), sum(255 - gt > 127), sum(gt * img > 127), sum((255 - gt) * img > 127)}, int64 products
__global__ void __launch_bounds__(256) tpr_fpr_kernel(const uint8_t* __restrict__ gt, const int64_t* __restrict__ img,
                                                     int64_t n, unsigned long long* __restrict__ counts4) {
    int pos = 0, neg = 0, tp = 0, fp = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t g = gt[e], v = img[e];
        pos += g > 127;
        neg += (255 - g) > 127;
        tp += (g * v) > 127;
        fp += ((255 - g) * v) > 127;
    }
    pos = __reduce_add_sync(0xffffffffu, pos); neg = __reduce_add_sync(0xffffffffu, neg);
    tp = __reduce_add_sync(0xffffffffu, tp); fp = __reduce_add_sync(0xffffffffu, fp);
    if ((threadIdx.x & 31) == 0) {
        if (pos) atomicAdd(counts4 + 0, (unsigned long long)pos);
        if (neg) atomicAdd(counts4 + 1, (unsigned long long)neg);
        if (tp) atomicAdd(counts4 + 2, (unsigned long long)tp);
        if (fp) atomicAdd(counts4 + 3, (unsigned long long)fp);
    }
}

int tpr_fpr_run(const uint8_t* d_gt, const int64_t* d_img, int64_t n, int64_t* d_counts4, cudaStream_t s) {
    MAVD_CUDA(cudaMemsetAsync(d_counts4, 0, 4 * sizeof(int64_t), s));
    tpr_fpr_kernel<<<148 * 4, 256, 0, s>>>(d_gt, d_img, n, reinterpret_cast<unsigned long long*>(d_counts4));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// 1-bit-per-pixel masks for the host<->device wire (include/mavd.h: mavd_pack_mask / mavd_unpack_mask).  The ground-truth
// segmentation going in and estimate_fixed coming out carry one bit of information per pixel; as byte masks they were
// two thirds of the bytes a batch moves over PCIe.  Thread = one 32-bit word = 32 pixels of the flattened frame, bit b
// of word j is pixel 32 j + b (numpy.packbits(..., bitorder='little')).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_mask_kernel(const uint8_t* __restrict__ mask, int64_t npx, int64_t words,
                                                       uint32_t* __restrict__ bits) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= words) return;
    const uint8_t* m = mask + (size_t)blockIdx.y * npx + 32 * j;
    uint32_t out = 0;
    if (32 * j + 32 <= npx && (reinterpret_cast<uintptr_t>(m) & 15) == 0) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(m)), b = __ldg(reinterpret_cast<const uint4*>(m) + 1);
        const uint32_t wv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            // one bit per non-zero byte, gathered into a nibble: the 0x01010101-masked word times 0x01020408 lands byte
            // k's bit at position 24 + k (no two partial products share a bit, so nothing carries)
            const uint32_t nz = __vcmpne4(wv[q], 0u) & 0x01010101u;
            out |= (((nz * 0x01020408u) >> 24) & 15u) << (4 * q);
        }
    } else {
        for (int b = 0; b < 32; ++b)
            if (32 * j + b < npx && m[b]) out |= 1u << b;
    }
    bits[(size_t)blockIdx.y * words + j] = out;
}

__global__ void __launch_bounds__(256) unpack_mask_kernel(const uint32_t* __restrict__ bits, int64_t npx, int64_t words,
                                                         uint32_t value, uint8_t* __restrict__ mask) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= words) return;
    const uint32_t v = __ldg(bits + (size_t)blockIdx.y * words + j);
    uint8_t* m = mask + (size_t)blockIdx.y * npx + 32 * j;
    if (32 * j + 32 <= npx && (reinterpret_cast<uintptr_t>(m) & 15) == 0) {
        uint32_t wv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint32_t nib = (v >> (4 * q)) & 15u;
            // spread the nibble's bits into the low bit of four bytes, then scale to `value`
            const uint32_t sp = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
            wv[q] = sp * value;
        }
        reinterpret_cast<uint4*>(m)[0] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        reinterpret_cast<uint4*>(m)[1] = make_uint4(wv[4], wv[5], wv[6], wv[7]);
    } else {
        for (int b = 0; b < 32; ++b)
            if (32 * j + b < npx) m[b] = (v >> b) & 1u ? (uint8_t)value : (uint8_t)0;
    }
}

int pack_mask_run(const uint8_t* d_mask, int n, int64_t npx, uint8_t* d_bits, cudaStream_t s) {
    const int64_t words = packed_mask_bytes(npx) / 4;
    pack_mask_kernel<<<dim3((unsigned)((words + 255) / 256), n), 256, 0, s>>>(d_mask, npx, words, (uint32_t*)d_bits);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

int unpack_mask_run(const uint8_t* d_bits, int n, int64_t npx, uint8_t value, uint8_t* d_mask, cudaStream_t s) {
    const int64_t words = packed_mask_bytes(npx) / 4;
    unpack_mask_kernel<<<dim3((unsigned)((words + 255) / 256), n), 256, 0, s>>>((const uint32_t*)d_bits, npx, words, value,
                                                                               d_mask);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Flow visualisation returned by Farneback.process() (farneback.py:83-99): cv2.cartToPolar -> hue/value bytes ->
// cv2.normalize(NORM_MINMAX) * 2 -> HSV2BGR.  The arithmetic restates what cv2 4.13 computes (verified
// bit-exact against cv2 on the CPU, see oracle/vis_np.py): magnitude sqrt(fma(x,x,y*y)); fastAtan2's degree-7
// polynomial evaluated with FMAs; float32 min-max normalisation; float->uint8 casts that truncate and wrap
// modulo 256 (NumPy's cast of the doubled value); 8-bit HSV2BGR with S = 255 through the float sector formula and
// a truncating store.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float cv_magnitude(float x, float y) { return __fsqrt_rn(__fmaf_rn(x, x, __fmul_rn(y, y))); }

__device__ __forceinline__ float cv_fast_atan2_rad(float y, float x) {
    const float p1 = 57.283627f, p3 = -18.667446f, p5 = 8.9140005f, p7 = -2.5397246f;
    const float ax = fabsf(x), ay = fabsf(y);
    const float mn = fminf(ax, ay), mx = fmaxf(ax, ay);
    const float c = __fdiv_rn(mn, __fadd_rn(mx, 2.220446049250313e-16f));
    const float c2 = __fmul_rn(c, c);
    float a = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmaf_rn(p7, c2, p5), c2, p3), c2, p1), c);
    if (ax < ay) a = __fsub_rn(90.f, a);
    if (x < 0.f) a = __fsub_rn(180.f, a);
    if (y < 0.f) a = __fsub_rn(360.f, a);
    return __fmul_rn(a, 0.017453292519943295f);
}

// scratch: [0] min(mag) bits, [1] max(mag) bits, [2] number of pixels whose value byte is non-zero
__global__ void vis_init_kernel(unsigned* scratch) {
    scratch[0] = 0x7f800000u;
    scratch[1] = 0u;
    scratch[2] = 0u;
}

__global__ void __launch_bounds__(256) vis_minmax_kernel(const float2* __restrict__ flow, int64_t n,
                                                        unsigned* __restrict__ scratch) {
    unsigned mn = 0x7f800000u, mx = 0u;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float2 v = flow[i];
        const unsigned b = __float_as_uint(cv_magnitude(v.x, v.y));   // magnitudes are >= 0: bit order == value order
        if (b <= 0x7f800000u) { mn = min(mn, b); mx = max(mx, b); }
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0) { atomicMin(scratch, mn); atomicMax(scratch + 1, mx); }
}

__device__ __forceinline__ unsigned f2u8_wrap(float v) {   // NumPy float32 -> uint8 assignment: truncate, wrap mod 256
    return (unsigned)((int)v) & 255u;
}

__global__ void __launch_bounds__(256) vis_kernel(const float2* __restrict__ flow, int64_t n, unsigned* __restrict__ scratch,
                                                 uint8_t* __restrict__ bgr) {
    const float mn = __uint_as_float(scratch[0]), mx = __uint_as_float(scratch[1]);
    // cv::normalize(NORM_MINMAX, 0..255): scale and shift in double, applied in float32
    const double span = (double)mx - (double)mn;
    const double dscale = 255.0 * (span > 2.220446049250313e-16 ? 1.0 / span : 0.0);
    const float scale = (float)dscale, shift = (float)(0.0 - (double)mn * dscale);
    int nz = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float2 f = flow[i];
        const float mag = cv_magnitude(f.x, f.y), ang = cv_fast_atan2_rad(f.y, f.x);
        unsigned h8 = f2u8_wrap(__fdiv_rn(__fdiv_rn(__fmul_rn(ang, 180.f), 3.14159274101257324f), 2.f));
        unsigned v8 = f2u8_wrap(__fmul_rn(__fadd_rn(__fmul_rn(mag, scale), shift), 2.f));
        nz += v8 != 0;
        if (v8 == 0) { h8 = 127; v8 = 255; }
        // HSV2BGR, S = 255
        const float v = __fmul_rn((float)v8, 1.f / 255.f);
        float h = __fmul_rn((float)h8, 6.f / 180.f);
        while (h >= 6.f) h = __fsub_rn(h, 6.f);
        int sec = (int)floorf(h);
        h = __fsub_rn(h, (float)sec);
        if ((unsigned)sec >= 6u) { sec = 0; h = 0.f; }
        float tab[4];
        tab[0] = v;
        tab[1] = __fmul_rn(v, 0.f);
        tab[2] = __fmul_rn(v, __fsub_rn(1.f, h));
        tab[3] = __fmul_rn(v, __fsub_rn(1.f, __fsub_rn(1.f, h)));
        const int sel = sec == 0 ? 0x130 : sec == 1 ? 0x102 : sec == 2 ? 0x301 : sec == 3 ? 0x021 : sec == 4 ? 0x013 : 0x210;
        const float b = tab[(sel >> 8) & 3], g = tab[(sel >> 4) & 3], r = tab[sel & 3];
        bgr[3 * i] = (uint8_t)min(255, max(0, (int)__fmul_rn(b, 255.f)));
        bgr[3 * i + 1] = (uint8_t)min(255, max(0, (int)__fmul_rn(g, 255.f)));
        bgr[3 * i + 2] = (uint8_t)min(255, max(0, (int)__fmul_rn(r, 255.f)));
    }
    nz = __reduce_add_sync(0xffffffffu, nz);
    if ((threadIdx.x & 31) == 0 && nz) atomicAdd(scratch + 2, (unsigned)nz);
}

int flow_vis_run(const float* d_flow, int64_t n, uint8_t* d_bgr, uint32_t* d_scratch3, cudaStream_t s) {
    vis_init_kernel<<<1, 1, 0, s>>>(d_scratch3);
    MAVD_LAUNCHED();
    vis_minmax_kernel<<<148 * 4, 256, 0, s>>>((const float2*)d_flow, n, d_scratch3);
    MAVD_LAUNCHED();
    vis_kernel<<<148 * 8, 256, 0, s>>>((const float2*)d_flow, n, d_scratch3, d_bgr);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Visualisation payloads of Processor.run_detection (next-row f4):
//   phi image      im_helpers.apply_colormap(im_helpers.to_rgb(phi, max_value=180)) — processor.py:324,376 with
//                  im_helpers.py:112-135,162-201: v = uint8(around(|phi| * 255 / max)) in phi's own dtype, GRAY2RGB, then
//                  cv2.applyColorMap(COLORMAP_JET), which for a 3-channel input takes BGR2GRAY (= v for equal
//                  channels) and looks v up in OpenCV's 256-entry JET table (embedded below, BGR order; pinned against
//                  cv2.applyColorMap in tests/test_oracle_vis.py)
//   mask overlay   mask_rgb = frame; mask_rgb[estimate_fixed] = (150, 0, 150);
//                  cv2.addWeighted(frame, 0.2, mask_rgb, 0.8, 0) — processor.py:385-392.  Unmasked pixels come out
//                  unchanged (0.2 v + 0.8 v rounds to v), masked ones are round(0.2 v + 0.8 c): 0.2 v is never within
//                  0.1 of a rounding tie, so the float evaluation order cannot matter.
// ------------------------------------------------------------------------------------------------
__constant__ uint8_t kJetLut[768] = {
    128, 0, 0, 132, 0, 0, 136, 0, 0, 140, 0, 0, 144, 0, 0, 148, 0, 0, 152, 0, 0, 156, 0, 0,
    160, 0, 0, 164, 0, 0, 168, 0, 0, 172, 0, 0, 176, 0, 0, 180, 0, 0, 184, 0, 0, 188, 0, 0,
    192, 0, 0, 196, 0, 0, 200, 0, 0, 204, 0, 0, 208, 0, 0, 212, 0, 0, 216, 0, 0, 220, 0, 0,
    224, 0, 0, 228, 0, 0, 232, 0, 0, 236, 0, 0, 240, 0, 0, 244, 0, 0, 248, 0, 0, 252, 0, 0,
    255, 0, 0, 255, 4, 0, 255, 8, 0, 255, 12, 0, 255, 16, 0, 255, 20, 0, 255, 24, 0, 255, 28, 0,
    255, 32, 0, 255, 36, 0, 255, 40, 0, 255, 44, 0, 255, 48, 0, 255, 52, 0, 255, 56, 0, 255, 60, 0,
    255, 64, 0, 255, 68, 0, 255, 72, 0, 255, 76, 0, 255, 80, 0, 255, 84, 0, 255, 88, 0, 255, 92, 0,
    255, 96, 0, 255, 100, 0, 255, 104, 0, 255, 108, 0, 255, 112, 0, 255, 116, 0, 255, 120, 0, 255, 124, 0,
    255, 128, 0, 255, 132, 0, 255, 136, 0, 255, 140, 0, 255, 144, 0, 255, 148, 0, 255, 152, 0, 255, 156, 0,
    255, 160, 0, 255, 164, 0, 255, 168, 0, 255, 172, 0, 255, 176, 0, 255, 180, 0, 255, 184, 0, 255, 188, 0,
    255, 192, 0, 255, 196, 0, 255, 200, 0, 255, 204, 0, 255, 208, 0, 255, 212, 0, 255, 216, 0, 255, 220, 0,
    255, 224, 0, 255, 228, 0, 255, 232, 0, 255, 236, 0, 255, 240, 0, 255, 244, 0, 255, 248, 0, 255, 252, 0,
    254, 255, 2, 250, 255, 6, 246, 255, 10, 242, 255, 14, 238, 255, 18, 234, 255, 22, 230, 255, 26, 226, 255, 30,
    222, 255, 34, 218, 255, 38, 214, 255, 42, 210, 255, 46, 206, 255, 50, 202, 255, 54, 198, 255, 58, 194, 255, 62,
    190, 255, 66, 186, 255, 70, 182, 255, 74, 178, 255, 78, 174, 255, 82, 170, 255, 86, 166, 255, 90, 162, 255, 94,
    158, 255, 98, 154, 255, 102, 150, 255, 106, 146, 255, 110, 142, 255, 114, 138, 255, 118, 134, 255, 122, 130, 255, 126,
    126, 255, 130, 122, 255, 134, 118, 255, 138, 114, 255, 142, 110, 255, 146, 106, 255, 150, 102, 255, 154, 98, 255, 158,
    94, 255, 162, 90, 255, 166, 86, 255, 170, 82, 255, 174, 78, 255, 178, 74, 255, 182, 70, 255, 186, 66, 255, 190,
    62, 255, 194, 58, 255, 198, 54, 255, 202, 50, 255, 206, 46, 255, 210, 42, 255, 214, 38, 255, 218, 34, 255, 222,
    30, 255, 226, 26, 255, 230, 22, 255, 234, 18, 255, 238, 14, 255, 242, 10, 255, 246, 6, 255, 250, 1, 255, 254,
    0, 252, 255, 0, 248, 255, 0, 244, 255, 0, 240, 255, 0, 236, 255, 0, 232, 255, 0, 228, 255, 0, 224, 255,
    0, 220, 255, 0, 216, 255, 0, 212, 255, 0, 208, 255, 0, 204, 255, 0, 200, 255, 0, 196, 255, 0, 192, 255,
    0, 188, 255, 0, 184, 255, 0, 180, 255, 0, 176, 255, 0, 172, 255, 0, 168, 255, 0, 164, 255, 0, 160, 255,
    0, 156, 255, 0, 152, 255, 0, 148, 255, 0, 144, 255, 0, 140, 255, 0, 136, 255, 0, 132, 255, 0, 128, 255,
    0, 124, 255, 0, 120, 255, 0, 116, 255, 0, 112, 255, 0, 108, 255, 0, 104, 255, 0, 100, 255, 0, 96, 255,
    0, 92, 255, 0, 88, 255, 0, 84, 255, 0, 80, 255, 0, 76, 255, 0, 72, 255, 0, 68, 255, 0, 64, 255,
    0, 60, 255, 0, 56, 255, 0, 52, 255, 0, 48, 255, 0, 44, 255, 0, 40, 255, 0, 36, 255, 0, 32, 255,
    0, 28, 255, 0, 24, 255, 0, 20, 255, 0, 16, 255, 0, 12, 255, 0, 8, 255, 0, 4, 255, 0, 0, 255,
    0, 0, 252, 0, 0, 248, 0, 0, 244, 0, 0, 240, 0, 0, 236, 0, 0, 232, 0, 0, 228, 0, 0, 224,
    0, 0, 220, 0, 0, 216, 0, 0, 212, 0, 0, 208, 0, 0, 204, 0, 0, 200, 0, 0, 196, 0, 0, 192,
    0, 0, 188, 0, 0, 184, 0, 0, 180, 0, 0, 176, 0, 0, 172, 0, 0, 168, 0, 0, 164, 0, 0, 160,
    0, 0, 156, 0, 0, 152, 0, 0, 148, 0, 0, 144, 0, 0, 140, 0, 0, 136, 0, 0, 132, 0, 0, 128,
};

template <typename T>
__global__ void __launch_bounds__(256) phi_colormap_kernel(const T* __restrict__ phi, int64_t n, T max_value,
                                                          uint8_t* __restrict__ gray_rgb, uint8_t* __restrict__ bgr) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const T a = phi[i] < T(0) ? -phi[i] : phi[i];
        unsigned v;
        if (sizeof(T) == 8) {
            const double t = __ddiv_rn(__dmul_rn((double)a, 255.0), (double)max_value);
            v = (t == t) ? ((unsigned)(long long)rint(t) & 255u) : 0u;        // around() is round-half-even
        } else {
            const float t = __fdiv_rn(__fmul_rn((float)a, 255.f), (float)max_value);
            v = (t == t) ? ((unsigned)(int)rintf(t) & 255u) : 0u;
        }
        if (gray_rgb) { gray_rgb[3 * i] = (uint8_t)v; gray_rgb[3 * i + 1] = (uint8_t)v; gray_rgb[3 * i + 2] = (uint8_t)v; }
        if (bgr) { bgr[3 * i] = kJetLut[3 * v]; bgr[3 * i + 1] = kJetLut[3 * v + 1]; bgr[3 * i + 2] = kJetLut[3 * v + 2]; }
    }
}

int phi_colormap_run(const void* d_phi, int is_f64, int64_t n, double max_value, uint8_t* d_gray_rgb, uint8_t* d_bgr,
                     cudaStream_t s) {
    if (!(max_value > 0.0)) max_value = 1.0;      // im_helpers.py:190-191
    const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 16);
    if (is_f64) phi_colormap_kernel<double><<<grid, 256, 0, s>>>((const double*)d_phi, n, max_value, d_gray_rgb, d_bgr);
    else phi_colormap_kernel<float><<<grid, 256, 0, s>>>((const float*)d_phi, n, (float)max_value, d_gray_rgb, d_bgr);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

__global__ void __launch_bounds__(256) mask_overlay_kernel(const uint8_t* __restrict__ frame, int channels,
                                                          const uint8_t* __restrict__ mask, int64_t n, uchar3 color,
                                                          float alpha, uint8_t* __restrict__ out,
                                                          uint8_t* __restrict__ mask_rgb) {
    const float beta = (float)(1.0 - (double)alpha);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint8_t px[3];
        if (channels == 3) { px[0] = frame[3 * i]; px[1] = frame[3 * i + 1]; px[2] = frame[3 * i + 2]; }
        else { px[0] = px[1] = px[2] = frame[i]; }
        const bool on = mask[i] != 0;
        const uint8_t c[3] = {color.x, color.y, color.z};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float other = on ? (float)c[k] : (float)px[k];
            const float t = __fadd_rn(__fmul_rn((float)px[k], alpha), __fmul_rn(other, beta));
            out[3 * i + k] = (uint8_t)min(255, max(0, (int)rintf(t)));      // cvRound + saturate_cast<uchar>
        }
        // im_helpers.to_rgb(255 * estimate_fixed) (processor.py:364): 0 / 255 on three equal channels
        if (mask_rgb) { const uint8_t m = on ? 255 : 0; mask_rgb[3 * i] = m; mask_rgb[3 * i + 1] = m; mask_rgb[3 * i + 2] = m; }
    }
}

int mask_overlay_run(const uint8_t* d_frame, int channels, const uint8_t* d_mask, int64_t n, uint8_t* d_out,
                     uint8_t* d_mask_rgb, cudaStream_t s) {
    const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 16);
    mask_overlay_kernel<<<grid, 256, 0, s>>>(d_frame, channels, d_mask, n, make_uchar3(150, 0, 150), 0.2f, d_out, d_mask_rgb);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// ------------------------------------------------------------------------------------------------
// Connected components (8-connectivity), union-find with the smaller raster index as the root, so a
// component's root is its first pixel in raster order and ranking the roots gives canonical labels.
//
// The passes never scan the image: they walk a LIST of occupied 128-pixel units (128 consecutive pixels of the
// flattened frame), one warp per unit.  The list is appended to by whoever produces the mask: residual_kernel while it
// writes the fixed mask (one atomic per occupied unit), or ccl_list_kernel, which streams a caller-supplied mask once.
//
// Everything is done on RUNS (maximal horizontal sequences of set pixels inside a unit and a row), not on pixels: the
// warp turns the unit into a 128-bit mask (four warp-uniform words, bit t of word j = pixel 32 j + t) and finds run
// starts / ends with shifts and bit scans.  Masks range from 0.1 % foreground (radial flow, a small mover) to 100 %
// (no FoE consensus, derotation mismatch): with one union per (run, neighbouring run) contact a dense 1080p frame
// costs ~2 unions per 128 pixels instead of ~2 per 4, only run starts walk the forest, and a component's box takes
// one update per run instead of five atomics per pixel (64 dense frames: 1.5 ms instead of 33 ms).
//   init     every set pixel points at the start of its run (depth 1, no memory traffic between pixels of a run)
//   merge    left contact (run at the unit's first pixel, previous pixel set), and for the row above: one union per
//            upper run that STARTS inside the run's 8-neighbourhood, one for an upper run that reaches it from the left
//   compress run starts halve their paths once more (stores allowed, the forest stays valid)
//   flatten  run starts point at their root (read-only walk: after the kernel boundary no halving store can undo it),
//            the other pixels copy their run start's root; roots are counted per unit
//   scan / rank / relabel as before: per-frame scan of the unit counts, rank of a root = canonical label
// A lane owns pixels t = 32 j + lane (j = 0..3) of the unit: parent / label accesses of a warp are 128-byte rows.
// ------------------------------------------------------------------------------------------------
// find with path halving (as in ECL-CC): every node passed on the way is re-pointed at its grandparent with a plain
// store.  Safe next to the concurrent atomicMin links of uf_union: a stored value is always an ancestor of the node
// (same set) with a smaller index (no cycles), and a link that such a store overwrites was only ever made redundant by
// uf_union continuing with the node's previous parent.
__device__ __forceinline__ int uf_find(int* parent, int i) {
    int cur = parent[i];
    if (cur != i) {
        int prev = i, next;
        while (cur > (next = parent[cur])) {
            parent[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

// read-only find for the flatten pass: there every run start is finally pointed at its ROOT, and a halving store from
// another thread landing after that write would leave it on a mere ancestor
__device__ __forceinline__ int uf_find_ro(const int* parent, int i) {
    int p = parent[i];
    while (p != i) {
        i = p;
        p = parent[i];
    }
    return i;
}

__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        const int old = atomicMin(parent + a, b);
        if (old == a) return;
        a = old;
    }
}

constexpr int CCL_UNIT = 128;                       // pixels per list entry
constexpr int CCL_GRID = 148 * 8;                   // blocks of 8 warps for the list passes

struct CclList {
    const int* entries;      // frame * n_units + unit, in no particular order
    const int* count;
    int n_units;             // units per frame
};

struct Bits128 { unsigned w[4]; };                  // bit t of w[j] = pixel 32 j + t (warp-uniform)

// The 128 mask pixels that start at frame pixel `start` (may be negative or run past the frame: those read as 0) as a
// warp-uniform bit mask.  VEC == 4 (width % 4 == 0, 4-byte aligned mask, start % 4 == 0): one 32-bit word per lane,
// nibbles gathered per group of eight lanes; VEC == 1: four byte loads per lane, one ballot each.
template <int VEC>
__device__ __forceinline__ Bits128 ccl_load_bits(const uint8_t* __restrict__ m, int start, int npx) {
    const int lane = threadIdx.x & 31;
    Bits128 b;
    if (VEC == 4) {
        const int px = start + 4 * lane;
        unsigned v = 0;
        if (px >= 0 && px + 4 <= npx) v = __ldg(reinterpret_cast<const unsigned*>(m + px));
        const unsigned nz = __vcmpne4(v, 0u) & 0x01010101u;
        const unsigned nib = ((nz * 0x01020408u) >> 24) & 15u;          // byte k non-zero -> bit k
        const unsigned grp = __reduce_or_sync(0xffu << (lane & 24), nib << (4 * (lane & 7)));
#pragma unroll
        for (int j = 0; j < 4; ++j) b.w[j] = __shfl_sync(0xffffffffu, grp, 8 * j);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int px = start + 32 * j + lane;
            const bool on = px >= 0 && px < npx && m[px] != 0;
            b.w[j] = __ballot_sync(0xffffffffu, on);
        }
    }
    return b;
}

__device__ __forceinline__ bool bit_of(const Bits128& b, int t) { return (b.w[t >> 5] >> (t & 31)) & 1u; }

// bit t of the result = bit t-1 of b (bit 0 = carry)
__device__ __forceinline__ Bits128 shl1(const Bits128& b, unsigned carry) {
    Bits128 r;
    r.w[0] = (b.w[0] << 1) | (carry & 1u);
#pragma unroll
    for (int j = 1; j < 4; ++j) r.w[j] = (b.w[j] << 1) | (b.w[j - 1] >> 31);
    return r;
}

// bit t of the result = bit t+1 of b (bit 127 = carry)
__device__ __forceinline__ Bits128 shr1(const Bits128& b, unsigned carry) {
    Bits128 r;
#pragma unroll
    for (int j = 0; j < 3; ++j) r.w[j] = (b.w[j] >> 1) | (b.w[j + 1] << 31);
    r.w[3] = (b.w[3] >> 1) | ((carry & 1u) << 31);
    return r;
}

// highest set bit of b at a position <= t (the caller guarantees there is one)
__device__ __forceinline__ int last_set_at_or_below(const Bits128& b, int t) {
    int j = t >> 5;
    unsigned w = b.w[j] & (0xffffffffu >> (31 - (t & 31)));
    while (w == 0 && j > 0) w = b.w[--j];
    return 32 * j + 31 - __clz(w);
}

// lowest set bit of b at a position >= t (the caller guarantees there is one)
__device__ __forceinline__ int first_set_at_or_above(const Bits128& b, int t) {
    int j = t >> 5;
    unsigned w = b.w[j] & (0xffffffffu << (t & 31));
    while (w == 0 && j < 3) w = b.w[++j];
    return 32 * j + __ffs(w) - 1;
}

// Geometry of one unit: which of its pixels begin a row (x == 0), run starts and run ends of its mask.
struct UnitRuns {
    Bits128 M, RS, S, E;     // mask, row starts, run starts, run ends
    int x0;                  // column of the unit's first pixel
};

__device__ __forceinline__ Bits128 row_starts(int ub, int w, int& x0_out) {
    const int lane = threadIdx.x & 31;
    const int x0 = ub % w;
    x0_out = x0;
    Bits128 rs;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int xt = (x0 + 32 * j + lane) % w;
        rs.w[j] = __ballot_sync(0xffffffffu, xt == 0);
    }
    return rs;
}

__device__ __forceinline__ void unit_runs(UnitRuns& R) {
    const Bits128 prev = shl1(R.M, 0u);                 // the pixel before the unit belongs to another unit's runs
    const Bits128 next = shr1(R.M, 0u), rs_next = shr1(R.RS, 1u);      // "pixel 128" always ends the run
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        R.S.w[j] = R.M.w[j] & (~prev.w[j] | R.RS.w[j]);
        R.E.w[j] = R.M.w[j] & (~next.w[j] | rs_next.w[j]);
    }
}

// list of occupied units of a caller-supplied mask (one streaming read); unit_mark doubles as the per-unit root count
// later, so only its zero / non-zero state matters here
template <int VEC>
__global__ void __launch_bounds__(256) ccl_list_kernel(const uint8_t* __restrict__ mask, int npx, int n_units, int n,
                                                      int* __restrict__ entries, int* __restrict__ count) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int total = n * n_units;
    for (int e = gw; e < total; e += warps) {
        const int f = e / n_units, u = e - f * n_units;
        const Bits128 b = ccl_load_bits<VEC>(mask + (size_t)f * npx, u * CCL_UNIT, npx);
        if ((b.w[0] | b.w[1] | b.w[2] | b.w[3]) && (threadIdx.x & 31) == 0) entries[atomicAdd(count, 1)] = e;
    }
}

// The row above a unit and the single pixels around it: U = the 128 pixels above the unit, um1 = the pixel before
// them, u128 = the pixel after them, prevpix = the pixel before the unit itself.
struct UnitAbove {
    Bits128 U, Uprev, US;    // upper pixels, upper pixels shifted by one (bit t = the pixel above t - 1), upper-run starts
    unsigned prevpix, um1, u128;
};

template <int VEC>
__device__ __forceinline__ UnitAbove unit_above(const uint8_t* __restrict__ m, int ub, int w, int npx, const Bits128& RS) {
    const int lane = threadIdx.x & 31;
    UnitAbove A;
    A.U = ccl_load_bits<VEC>(m, ub - w, npx);
    unsigned side = 0;
    if (lane == 0 && ub >= 1) side = m[ub - 1] != 0;
    if (lane == 1 && ub - w - 1 >= 0) side = m[ub - w - 1] != 0;
    if (lane == 2 && ub - w + CCL_UNIT >= 0 && ub - w + CCL_UNIT < npx) side = m[ub - w + CCL_UNIT] != 0;
    const unsigned sides = __ballot_sync(0xffffffffu, side != 0);
    A.prevpix = sides & 1u; A.um1 = (sides >> 1) & 1u; A.u128 = (sides >> 2) & 1u;
    A.Uprev = shl1(A.U, A.um1);
#pragma unroll
    for (int j = 0; j < 4; ++j) A.US.w[j] = A.U.w[j] & (~A.Uprev.w[j] | RS.w[j]);   // a row start always starts a run
    return A;
}

// init: every set pixel points at the start of its run inside the unit.  A run that continues one ending the previous
// unit (same row) is linked to it right here, without an atomic: its start points at the previous pixel (smaller
// index, same component).  These chains are at most two hops per unit of a row, and they remove half of the unions of
// a densely set frame; contacts with the row above stay with the merge pass (linking them here as well was measured:
// it builds image-high chains that the later passes pay for).
template <int VEC>
__global__ void __launch_bounds__(256) ccl_init_kernel(const uint8_t* __restrict__ mask, int* __restrict__ parent, int w,
                                                      int npx, CclList L) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        const uint8_t* m = mask + (size_t)f * npx;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(m, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        const bool left_cont = (R.M.w[0] & 1u) && !(R.RS.w[0] & 1u) && ub >= 1 && m[ub - 1] != 0;   // warp-uniform
        int* par = parent + (size_t)f * npx;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int t = 32 * j + lane;
            if (!((R.M.w[j] >> lane) & 1u)) continue;
            const int s = last_set_at_or_below(R.S, t);
            par[ub + t] = (t == 0 && left_cont) ? ub - 1 : ub + s;
        }
    }
}

// merge: one union per contact between a run [s, e] of this unit and a run of the row above:
//   (B)  the upper run covers column s - 1 (it started at or before s - 1): one union at s — unless the run continues
//        from the previous unit, whose last pixel has that same upper run above it and has taken care of it
//   (A)  an upper run STARTS at a column t in [s, e + 1]: one union, by the lane that owns t (with pixel t if it is
//        set, else with pixel t - 1, whose up-right neighbour it is); a start at column 128 by pixel 127's owner
// A fully set frame makes one union per image row.
template <int VEC>
__global__ void __launch_bounds__(256) ccl_merge_kernel(const uint8_t* __restrict__ mask, int* __restrict__ parent, int w,
                                                       int npx, CclList L) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        const uint8_t* m = mask + (size_t)f * npx;
        int* par = parent + (size_t)f * npx;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(m, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        const UnitAbove A = unit_above<VEC>(m, ub, w, npx, R.RS);
        if (!(A.U.w[0] | A.U.w[1] | A.U.w[2] | A.U.w[3] | A.um1 | A.u128)) continue;    // nothing above: warp-uniform
        const bool left_cont = A.prevpix && !(R.RS.w[0] & 1u) && (R.M.w[0] & 1u);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int t = 32 * j + lane, g = ub + t;
            const bool mt = (R.M.w[j] >> lane) & 1u, rs = (R.RS.w[j] >> lane) & 1u;
            if (mt && ((R.S.w[j] >> lane) & 1u) && !rs && !(t == 0 && left_cont) && ((A.Uprev.w[j] >> lane) & 1u))
                uf_union(par, g, g - w - 1);                                                      // (B)
            if ((A.US.w[j] >> lane) & 1u) {                                                       // (A)
                if (mt) uf_union(par, g, g - w);
                else if (t >= 1 && !rs && bit_of(R.M, t - 1)) uf_union(par, g - 1, g - w);
            }
            if (t == CCL_UNIT - 1 && mt && A.u128 && !((A.U.w[3] >> 31) & 1u) && (R.x0 + CCL_UNIT) % w != 0)
                uf_union(par, g, g - w + 1);
        }
    }
}

// run starts halve their paths once more before the read-only flatten
template <int VEC>
__global__ void __launch_bounds__(256) ccl_compress_kernel(const uint8_t* __restrict__ mask, int* __restrict__ parent, int w,
                                                          int npx, CclList L) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + (size_t)f * npx, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        int* par = parent + (size_t)f * npx;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if ((R.S.w[j] >> lane) & 1u) uf_find(par, ub + 32 * j + lane);
    }
}

// flatten + count the roots of every listed unit (unit_cnt[e]; units that are not listed keep their zero)
template <int VEC>
__global__ void __launch_bounds__(256) ccl_flatten_count_kernel(const uint8_t* __restrict__ mask, int* __restrict__ parent,
                                                               int w, int npx, CclList L, int* __restrict__ unit_cnt) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + (size_t)f * npx, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        int* par = parent + (size_t)f * npx;
        int roots = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (!((R.S.w[j] >> lane) & 1u)) continue;
            const int g = ub + 32 * j + lane;
            const int r = uf_find_ro(par, g);
            par[g] = r;      // benign race with other walkers: whoever reads it sees an ancestor or the root
            roots += (r == g);
        }
        __syncwarp();
        // the other pixels of a run take their run start's root (written above by a lane of this warp)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int t = 32 * j + lane;
            if (((R.M.w[j] & ~R.S.w[j]) >> lane) & 1u) par[ub + t] = par[ub + last_set_at_or_below(R.S, t)];
        }
        roots = __reduce_add_sync(0xffffffffu, roots);
        if (lane == 0) unit_cnt[e] = roots;     // overwrites the producer's "listed" mark
    }
}

// exclusive scan of the per-unit root counts, one block per frame; writes the total label count
__global__ void __launch_bounds__(1024) ccl_scan_kernel(int* __restrict__ unit_cnt, int n_units, char* nlabels_base,
                                                       size_t nlabels_stride) {
    pdl_entry();
    __shared__ int wtot[32];
    __shared__ int carry_s;
    int* c = unit_cnt + (size_t)blockIdx.x * n_units;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    // 4 consecutive units per thread: a 1080p frame (16 200 units) is four rounds
    for (int base = 0; base < n_units; base += 4096) {
        const int i = base + threadIdx.x * 4;
        int v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = i + k < n_units ? c[i + k] : 0;
        const int mine = v[0] + v[1] + v[2] + v[3];
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wtot[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            int wv = wtot[lane], wi = wv;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            wtot[lane] = wi - wv;
        }
        __syncthreads();
        const int carry = carry_s;
        int off = carry + wtot[wid] + incl - mine;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (i + k < n_units) c[i + k] = off;
            off += v[k];
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = off;
        __syncthreads();
    }
    if (threadIdx.x == 0) *reinterpret_cast<int32_t*>(nlabels_base + (size_t)blockIdx.x * nlabels_stride) = carry_s;
}

// rank[root] = canonical label of the component rooted at `root` (roots ordered by raster index): the unit's offset
// from the scan plus the raster-order prefix inside the unit
template <int VEC>
__global__ void __launch_bounds__(256) ccl_rank_kernel(const uint8_t* __restrict__ mask, const int* __restrict__ parent,
                                                      int w, int npx, CclList L, const int* __restrict__ unit_off,
                                                      int* __restrict__ rank) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + (size_t)f * npx, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        const int* par = parent + (size_t)f * npx;
        int* rk = rank + (size_t)f * npx;
        int running = unit_off[e];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int g = ub + 32 * j + lane;
            const bool root = ((R.S.w[j] >> lane) & 1u) && par[g] == g;
            const unsigned roots = __ballot_sync(0xffffffffu, root);
            if (root) rk[g] = running + __popc(roots & ((1u << lane) - 1u)) + 1;
            running += __popc(roots);
        }
    }
}

__global__ void ccl_boxes_init_kernel(int32_t* boxes, size_t boxes_stride, int max_boxes, int n) {
    pdl_entry();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * max_boxes) return;
    int f = i / max_boxes, b = i - f * max_boxes;
    int32_t* p = boxes + (size_t)f * boxes_stride + b * 5;
    p[0] = 0x7fffffff; p[1] = 0x7fffffff; p[2] = -1; p[3] = -1; p[4] = 0;
}

// labels_out may alias parent: a warp reads only the parent entries of its own unit's run starts, all before its
// first label store; background pixels were zeroed before the init pass.
// Boxes: one contribution per RUN.  A warp walks ~100 units; consecutive list entries mostly belong to the same frame
// and, in dense masks, to the same component, whose five box words would otherwise take an atomic per run from every
// warp at once.  So the warp keeps ONE (frame, label) box in registers: runs of that label are folded in with warp
// reductions, the box is flushed (five atomics by one lane) only when the unit's first label changes; runs of other
// labels in the unit go out directly, bounds first checked against the current value (monotone: a stale read can only
// cause a redundant atomic, never a missed one).
struct BoxAcc {
    int key = -1;            // frame * (max_boxes + 1) + label, -1 = empty
    int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1, area = 0;
};

__device__ __forceinline__ void box_flush(BoxAcc& acc, int32_t* boxes, size_t boxes_stride, int max_boxes) {
    if (acc.key >= 0 && acc.area > 0 && (threadIdx.x & 31) == 0) {
        const int f = acc.key / (max_boxes + 1), l = acc.key - f * (max_boxes + 1);
        int32_t* bx = boxes + (size_t)f * boxes_stride + (l - 1) * 5;
        atomicMin(bx + 0, acc.x0); atomicMin(bx + 1, acc.y0); atomicMax(bx + 2, acc.x1); atomicMax(bx + 3, acc.y1);
        atomicAdd(bx + 4, acc.area);
    }
    acc = BoxAcc();
}

template <int VEC>
__global__ void __launch_bounds__(256) ccl_relabel_kernel(const uint8_t* __restrict__ mask, const int* parent,
                                                         const int* __restrict__ rank, int w, int npx, CclList L,
                                                         int* labels_out, int32_t* boxes,
                                                         size_t boxes_stride, int max_boxes) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const int cnt = *L.count;
    BoxAcc acc;
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        const size_t base = (size_t)f * npx;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + base, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        int lab[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            lab[j] = 0;
            if ((R.S.w[j] >> lane) & 1u) lab[j] = rank[base + parent[base + ub + 32 * j + lane]];
        }
        if (boxes) {
            // the unit's first run decides which label the warp accumulates
            const int s0 = first_set_at_or_above(R.S, 0);
            int l0 = 0;
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int v = __shfl_sync(FULL, lab[jj], s0 & 31);
                if ((s0 >> 5) == jj) l0 = v;
            }
            const int key0 = l0 <= max_boxes ? f * (max_boxes + 1) + l0 : -1;
            if (key0 != acc.key) {
                box_flush(acc, boxes, boxes_stride, max_boxes);
                acc.key = key0;
            }
            int ax0 = 0x7fffffff, ay0 = 0x7fffffff, ax1 = -1, ay1 = -1, aarea = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (!((R.S.w[j] >> lane) & 1u)) continue;
                const int l = lab[j];
                if (l > max_boxes) continue;
                const int t = 32 * j + lane, g = ub + t;
                const int len = first_set_at_or_above(R.E, t) - t + 1;
                const int y = g / w, xs = g - y * w, xe = xs + len - 1;
                if (l == l0 && key0 >= 0) {
                    ax0 = min(ax0, xs); ay0 = min(ay0, y); ax1 = max(ax1, xe); ay1 = max(ay1, y); aarea += len;
                } else {
                    int32_t* bx = boxes + (size_t)f * boxes_stride + (l - 1) * 5;
                    if (xs < __ldcg(bx + 0)) atomicMin(bx + 0, xs);
                    if (y < __ldcg(bx + 1)) atomicMin(bx + 1, y);
                    if (xe > __ldcg(bx + 2)) atomicMax(bx + 2, xe);
                    if (y > __ldcg(bx + 3)) atomicMax(bx + 3, y);
                    atomicAdd(bx + 4, len);
                }
            }
            if (key0 >= 0) {
                acc.x0 = min(acc.x0, __reduce_min_sync(FULL, ax0)); acc.y0 = min(acc.y0, __reduce_min_sync(FULL, ay0));
                acc.x1 = max(acc.x1, __reduce_max_sync(FULL, ax1)); acc.y1 = max(acc.y1, __reduce_max_sync(FULL, ay1));
                acc.area += __reduce_add_sync(FULL, aarea);
            }
        }
        if (labels_out) {
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = 32 * j + lane;
                const bool on = (R.M.w[j] >> lane) & 1u;
                const int s = on ? last_set_at_or_below(R.S, t) : 0;
                int l = 0;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int v = __shfl_sync(FULL, lab[jj], s & 31);
                    if ((s >> 5) == jj) l = v;
                }
                if (on) labels_out[base + ub + t] = l;
            }
        }
    }
    if (boxes) box_flush(acc, boxes, boxes_stride, max_boxes);
}

__global__ void ccl_boxes_final_kernel(int32_t* boxes, size_t boxes_stride, int max_boxes, int n) {
    pdl_entry();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * max_boxes) return;
    int f = i / max_boxes, b = i - f * max_boxes;
    int32_t* p = boxes + (size_t)f * boxes_stride + b * 5;
    if (p[4] == 0) { p[0] = p[1] = p[2] = p[3] = 0; }
    else { p[2] = p[2] - p[0] + 1; p[3] = p[3] - p[1] + 1; }
}

// ------------------------------------------------------------------------------------------------
// Detection tables (mavd_detection): the max_det largest components of every frame, from the same unit list, forest
// and rank array that give the record's boxes.
//   zero    the per-label areas of labels 1..n_labels
//   area    pass A: area of every label, runs of one label folded in registers (the BoxAcc pattern)
//   select  one CTA per frame: exact top max_det by (area desc, label asc) — radix select of the cut-off area over
//           10-bit digits, ties at the cut taken in label order — then lab_area[label] = -(slot + 1) for the selected
//           labels and every table entry initialised
//   stats   pass B: box, area, index sums and derotated flow of the selected labels only
//   final   box corners -> width / height
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) det_area_zero_kernel(int32_t* __restrict__ lab_area, int lab_stride,
                                                            const char* nlabels_base, size_t nlabels_stride) {
    pdl_entry();
    const int f = blockIdx.y;
    const int nl = *reinterpret_cast<const int32_t*>(nlabels_base + (size_t)f * nlabels_stride);
    int32_t* A = lab_area + (size_t)f * lab_stride;
    for (int l = blockIdx.x * blockDim.x + threadIdx.x; l <= nl; l += gridDim.x * blockDim.x) A[l] = 0;
}

// label of every run start of the unit (0 elsewhere) and the label of the unit's first run (warp-uniform)
__device__ __forceinline__ int unit_labels(const UnitRuns& R, const int* parent, const int* __restrict__ rank, size_t base,
                                           int ub, int lab[4]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        lab[j] = 0;
        if ((R.S.w[j] >> lane) & 1u) lab[j] = rank[base + parent[base + ub + 32 * j + lane]];
    }
    const int s0 = first_set_at_or_above(R.S, 0);
    int l0 = 0;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const int v = __shfl_sync(0xffffffffu, lab[jj], s0 & 31);
        if ((s0 >> 5) == jj) l0 = v;
    }
    return l0;
}

template <int VEC>
__global__ void __launch_bounds__(256) det_area_kernel(const uint8_t* __restrict__ mask, const int* parent,
                                                       const int* __restrict__ rank, int w, int npx, CclList L,
                                                       int32_t* __restrict__ lab_area, int lab_stride) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int cnt = *L.count;
    int acc_f = -1, acc_l = 0, acc_area = 0;       // the (frame, label) whose area the warp holds in registers
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        const size_t base = (size_t)f * npx;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + base, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        int lab[4];
        const int l0 = unit_labels(R, parent, rank, base, ub, lab);
        if (f != acc_f || l0 != acc_l) {
            if (acc_f >= 0 && lane == 0) atomicAdd(lab_area + (size_t)acc_f * lab_stride + acc_l, acc_area);
            acc_f = f; acc_l = l0; acc_area = 0;
        }
        int mine = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (!((R.S.w[j] >> lane) & 1u)) continue;
            const int t = 32 * j + lane;
            const int len = first_set_at_or_above(R.E, t) - t + 1;
            if (lab[j] == l0) mine += len;
            else atomicAdd(lab_area + (size_t)f * lab_stride + lab[j], len);
        }
        acc_area += __reduce_add_sync(0xffffffffu, mine);
    }
    if (acc_f >= 0 && lane == 0) atomicAdd(lab_area + (size_t)acc_f * lab_stride + acc_l, acc_area);
}

// exclusive prefix of v over the 1024 threads of the block; *total receives the sum (wtot: 33 ints of shared memory,
// free again when the function returns)
__device__ __forceinline__ int block_excl_scan_1024(int v, int* wtot, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wtot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        const int wv = wtot[lane];
        int wi = wv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        wtot[lane] = wi - wv;
        if (lane == 31) wtot[32] = wi;
    }
    __syncthreads();
    const int r = wtot[wid] + incl - v;
    *total = wtot[32];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(1024) det_select_kernel(int32_t* __restrict__ lab_area, int lab_stride,
                                                          const char* nlabels_base, size_t nlabels_stride,
                                                          mavd_detection* __restrict__ det, int max_det) {
    pdl_entry();
    __shared__ int hist[1024];
    __shared__ int wtot[33];
    __shared__ int sel_lab[MAVD_MAX_DETECTIONS], sel_area[MAVD_MAX_DETECTIONS];
    __shared__ int s_digit, s_above, s_cnt;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int nl = *reinterpret_cast<const int32_t*>(nlabels_base + (size_t)f * nlabels_stride);
    int32_t* A = lab_area + (size_t)f * lab_stride;
    // every label with area > cut is taken, and the first take_eq labels with area == cut; with at most max_det labels
    // all are taken (every label has an area >= 1)
    int cut = 0, take_eq = 0;
    if (nl > max_det) {
        int prefix = 0, hi_mask = 0, rem = max_det;   // rem-th largest area among the labels that match the prefix
        for (int shift = 20; shift >= 0; shift -= 10) {    // areas < 2^28 (16384^2 pixels)
            hist[tid] = 0;
            __syncthreads();
            for (int l = 1 + tid; l <= nl; l += 1024) {
                const int a = A[l];
                if ((a & hi_mask) == prefix) atomicAdd(&hist[(a >> shift) & 1023], 1);
            }
            __syncthreads();
            // thread t looks at digit 1023 - t: inclusive prefix = labels with that digit or a larger one
            const int c = hist[1023 - tid];
            int tot;
            const int ex = block_excl_scan_1024(c, wtot, &tot);
            if (ex < rem && ex + c >= rem) { s_digit = 1023 - tid; s_above = ex; }
            __syncthreads();
            prefix |= s_digit << shift;
            hi_mask |= 1023 << shift;
            rem -= s_above;
            __syncthreads();
        }
        cut = prefix;
        take_eq = rem;
    }
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    int eq_seen = 0;
    for (int b = 1; b <= nl; b += 1024) {
        const int l = b + tid;
        const int a = l <= nl ? A[l] : 0;
        const bool eq = a == cut && a > 0;
        int tot;
        const int r = block_excl_scan_1024(eq ? 1 : 0, wtot, &tot);
        if (a > cut || (eq && eq_seen + r < take_eq)) {
            const int pos = atomicAdd(&s_cnt, 1);
            sel_lab[pos] = l;
            sel_area[pos] = a;
        }
        eq_seen += tot;
    }
    __syncthreads();
    const int cnt = s_cnt;     // == min(nl, max_det)
    mavd_detection* D = det + (size_t)f * max_det;
    for (int i = tid; i < max_det; i += 1024) {
        if (i < cnt) {
            const int a = sel_area[i], l = sel_lab[i];
            int r = 0;
            for (int k = 0; k < cnt; ++k) r += sel_area[k] > a || (sel_area[k] == a && sel_lab[k] < l);
            mavd_detection& d = D[r];
            d.label = l;
            d.box[0] = 0x7fffffff; d.box[1] = 0x7fffffff; d.box[2] = -1; d.box[3] = -1;
            d.area = 0;
            d.sum_x = 0; d.sum_y = 0;
            d.flow_sum[0] = 0.0; d.flow_sum[1] = 0.0;
            A[l] = -(r + 1);
        }
        if (i >= cnt) {
            mavd_detection& d = D[i];
            d.label = 0;
            d.box[0] = d.box[1] = d.box[2] = d.box[3] = 0;
            d.area = 0;
            d.sum_x = 0; d.sum_y = 0;
            d.flow_sum[0] = 0.0; d.flow_sum[1] = 0.0;
        }
    }
}

// Statistics of one table entry accumulated by a warp (runs of the entry the unit starts with) before one flush.
struct DetAcc {
    int f = -1, slot = -1;
    int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1, area = 0;
    long long sx = 0, sy = 0;
    double fx = 0.0, fy = 0.0;
};

__device__ __forceinline__ void det_flush(DetAcc& acc, mavd_detection* det, int max_det) {
    if (acc.f >= 0 && acc.area > 0 && (threadIdx.x & 31) == 0) {
        mavd_detection* d = det + (size_t)acc.f * max_det + acc.slot;
        atomicMin(&d->box[0], acc.x0); atomicMin(&d->box[1], acc.y0);
        atomicMax(&d->box[2], acc.x1); atomicMax(&d->box[3], acc.y1);
        atomicAdd(&d->area, acc.area);
        atomicAdd(reinterpret_cast<unsigned long long*>(&d->sum_x), (unsigned long long)acc.sx);
        atomicAdd(reinterpret_cast<unsigned long long*>(&d->sum_y), (unsigned long long)acc.sy);
        atomicAdd(&d->flow_sum[0], acc.fx);
        atomicAdd(&d->flow_sum[1], acc.fy);
    }
    acc = DetAcc();
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int VEC>
__global__ void __launch_bounds__(256) det_stats_kernel(const uint8_t* __restrict__ mask, const int* parent,
                                                        const int* __restrict__ rank, int w, int h, int npx, CclList L,
                                                        const int32_t* __restrict__ lab_area, int lab_stride,
                                                        const float* __restrict__ flow, const mavd_imu* __restrict__ imu,
                                                        mavd_detection* det, int max_det) {
    pdl_entry();
    const int warps = gridDim.x * 8, gw = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const int cnt = *L.count;
    DetAcc acc;
    int derot_f = -1;
    Derot D{};
    for (int q = gw; q < cnt; q += warps) {
        const int e = L.entries[q];
        const int f = e / L.n_units, u = e - f * L.n_units, ub = u * CCL_UNIT;
        const size_t base = (size_t)f * npx;
        UnitRuns R;
        R.M = ccl_load_bits<VEC>(mask + base, ub, npx);
        R.RS = row_starts(ub, w, R.x0);
        unit_runs(R);
        int lab[4], sl[4];
        const int l0 = unit_labels(R, parent, rank, base, ub, lab);
        bool any = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            sl[j] = -1;
            if (lab[j] > 0) {
                const int v = lab_area[(size_t)f * lab_stride + lab[j]];
                if (v < 0) sl[j] = -v - 1;
            }
            any |= sl[j] >= 0;
        }
        if (!__any_sync(FULL, any)) continue;                 // no selected component in this unit
        const int m0 = lab_area[(size_t)f * lab_stride + l0];
        const int slot0 = m0 < 0 ? -m0 - 1 : -1;             // the entry the warp accumulates in registers
        if (slot0 >= 0 && (f != acc.f || slot0 != acc.slot)) {
            det_flush(acc, det, max_det);
            acc.f = f; acc.slot = slot0;
        }
        int ax0 = 0x7fffffff, ay0 = 0x7fffffff, ax1 = -1, ay1 = -1, aarea = 0, asx = 0, asy = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (sl[j] < 0) continue;
            const int t = 32 * j + lane, g = ub + t;
            const int len = first_set_at_or_above(R.E, t) - t + 1;
            const int y = g / w, xs = g - y * w, xe = xs + len - 1;
            const int sx = len * xs + len * (len - 1) / 2, sy = len * y;    // < 128 * 16384: no overflow
            if (sl[j] == slot0) {
                ax0 = min(ax0, xs); ay0 = min(ay0, y); ax1 = max(ax1, xe); ay1 = max(ay1, y);
                aarea += len; asx += sx; asy += sy;
            } else {
                mavd_detection* d = det + (size_t)f * max_det + sl[j];
                atomicMin(&d->box[0], xs); atomicMin(&d->box[1], y); atomicMax(&d->box[2], xe); atomicMax(&d->box[3], y);
                atomicAdd(&d->area, len);
                atomicAdd(reinterpret_cast<unsigned long long*>(&d->sum_x), (unsigned long long)sx);
                atomicAdd(reinterpret_cast<unsigned long long*>(&d->sum_y), (unsigned long long)sy);
            }
        }
        double fx = 0.0, fy = 0.0;
        if (flow) {
            if (f != derot_f) { D = make_derot(imu[f], w, h); derot_f = f; }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int t = 32 * j + lane;
                const bool on = (R.M.w[j] >> lane) & 1u;
                const int s = on ? last_set_at_or_below(R.S, t) : 0;
                int ps = -1;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int v = __shfl_sync(FULL, sl[jj], s & 31);
                    if ((s >> 5) == jj) ps = v;
                }
                if (!on || ps < 0) continue;
                const int g = ub + t, y = g / w, x = g - y * w;
                const float* p = flow + 2 * (base + g);
                double v0 = (double)__ldg(p), v1 = (double)__ldg(p + 1);
                if (D.on) {
                    double r0, r1;
                    derot_at(D, x, y, r0, r1);
                    v0 = __dsub_rn(v0, r0);
                    v1 = __dsub_rn(v1, r1);
                }
                if (ps == slot0) {
                    fx = __dadd_rn(fx, v0);
                    fy = __dadd_rn(fy, v1);
                } else {
                    mavd_detection* d = det + (size_t)f * max_det + ps;
                    atomicAdd(&d->flow_sum[0], v0);
                    atomicAdd(&d->flow_sum[1], v1);
                }
            }
        }
        if (slot0 >= 0) {
            acc.x0 = min(acc.x0, __reduce_min_sync(FULL, ax0)); acc.y0 = min(acc.y0, __reduce_min_sync(FULL, ay0));
            acc.x1 = max(acc.x1, __reduce_max_sync(FULL, ax1)); acc.y1 = max(acc.y1, __reduce_max_sync(FULL, ay1));
            acc.area += __reduce_add_sync(FULL, aarea);
            acc.sx += __reduce_add_sync(FULL, asx);
            acc.sy += __reduce_add_sync(FULL, asy);
            if (flow) {
                acc.fx += warp_sum_f64(fx);
                acc.fy += warp_sum_f64(fy);
            }
        }
    }
    det_flush(acc, det, max_det);
}

__global__ void det_final_kernel(mavd_detection* det, int total) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    mavd_detection& d = det[i];
    if (d.label == 0) return;
    d.box[2] = d.box[2] - d.box[0] + 1;
    d.box[3] = d.box[3] - d.box[1] + 1;
}

// scratch behind the rank array: [count (4 ints)] [unit_cnt: max_pairs x n_units] [entries: max_pairs x n_units]
int ccl_n_units(mavd_handle H) { return ceil_div(H->cfg.width * H->cfg.height, CCL_UNIT); }
static int* ccl_count_ptr(mavd_handle H) { return H->d_scan + (size_t)H->cfg.max_pairs * H->cfg.width * H->cfg.height; }
int* ccl_unit_marks(mavd_handle H) { return ccl_count_ptr(H) + 4; }
int* ccl_unit_list(mavd_handle H) { return ccl_unit_marks(H) + (size_t)H->cfg.max_pairs * ccl_n_units(H); }
int* ccl_unit_count(mavd_handle H) { return ccl_count_ptr(H); }

// zeroes the list counter and the per-unit marks of n frames (a kernel, not a memset: it stays inside the chain of
// programmatic dependent launches, common.cuh)
__global__ void __launch_bounds__(256) ccl_list_reset_kernel(int* __restrict__ p, size_t n_ints) {
    pdl_entry();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_ints; i += stride) p[i] = 0;
}

int ccl_list_reset(mavd_handle H, int n, cudaStream_t s, int lane) {
    const size_t n_ints = 4 + (size_t)n * ccl_n_units(H);
    const int blocks = (int)min((size_t)148 * 8, (n_ints + 255) / 256);
    MAVD_CUDA(launch_chained(pdl_next(H, lane), ccl_list_reset_kernel, blocks, 256, 0, s, ccl_count_ptr(H), n_ints));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

template <int VEC>
static int ccl_launch(mavd_handle H, const uint8_t* d_mask, int n, int* parent, int32_t* labels_out, int32_t* d_boxes,
                      size_t boxes_stride, int max_boxes, int32_t* d_n_labels, size_t nlabels_stride, cudaStream_t s,
                      bool list_ready, const DetArgs* det) {
    const int w = H->cfg.width, h = H->cfg.height, npx = w * h;
    const int n_units = ccl_n_units(H);
    int* rank = H->d_scan;                     // [n][npx], written and read at roots only
    int* unit_cnt = ccl_unit_marks(H);         // [n][n_units]: "listed" mark, then root count, then label offset
    CclList L{ccl_unit_list(H), ccl_unit_count(H), n_units};
    if (!list_ready) {
        TRY_RC(ccl_list_reset(H, n, s));
        MAVD_CUDA(launch_chained(pdl_next(H), ccl_list_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, npx, n_units, n,
                                 ccl_unit_list(H), ccl_unit_count(H)));
        MAVD_LAUNCHED();
    }
    if (labels_out) {
        MAVD_CUDA(cudaMemsetAsync(labels_out, 0, sizeof(int32_t) * (size_t)n * npx, s));
        pdl_break(H);
    }
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_init_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, w, npx, L));
    MAVD_LAUNCHED();
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_merge_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, w, npx, L));
    MAVD_LAUNCHED();
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_compress_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, w, npx, L));
    MAVD_LAUNCHED();
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_flatten_count_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, w, npx, L, unit_cnt));
    MAVD_LAUNCHED();
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_scan_kernel, n, 1024, 0, s, unit_cnt, n_units, (char*)d_n_labels, nlabels_stride));
    MAVD_LAUNCHED();
    MAVD_CUDA(launch_chained(pdl_next(H), ccl_rank_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, w, npx, L, unit_cnt, rank));
    MAVD_LAUNCHED();
    if (d_boxes) {
        MAVD_CUDA(launch_chained(pdl_next(H), ccl_boxes_init_kernel, ceil_div(n * max_boxes, 128), 128, 0, s, d_boxes,
                                 boxes_stride, max_boxes, n));
        MAVD_LAUNCHED();
    }
    if (d_boxes || labels_out) {
        MAVD_CUDA(launch_chained(pdl_next(H), ccl_relabel_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, rank, w, npx, L,
                                 labels_out, d_boxes, boxes_stride, max_boxes));
        MAVD_LAUNCHED();
    }
    if (d_boxes) {
        MAVD_CUDA(launch_chained(pdl_next(H), ccl_boxes_final_kernel, ceil_div(n * max_boxes, 128), 128, 0, s, d_boxes,
                                 boxes_stride, max_boxes, n));
        MAVD_LAUNCHED();
    }
    if (det) {
        const char* nl = reinterpret_cast<const char*>(d_n_labels);
        MAVD_CUDA(launch_chained(pdl_next(H), det_area_zero_kernel, dim3(ceil_div(det->lab_stride, 256 * 8), n), 256, 0, s,
                                 det->lab_area, det->lab_stride, nl, nlabels_stride));
        MAVD_LAUNCHED();
        MAVD_CUDA(launch_chained(pdl_next(H), det_area_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, rank, w, npx, L,
                                 det->lab_area, det->lab_stride));
        MAVD_LAUNCHED();
        MAVD_CUDA(launch_chained(pdl_next(H), det_select_kernel, n, 1024, 0, s, det->lab_area, det->lab_stride, nl,
                                 nlabels_stride, det->det, det->max_det));
        MAVD_LAUNCHED();
        MAVD_CUDA(launch_chained(pdl_next(H), det_stats_kernel<VEC>, CCL_GRID, 256, 0, s, d_mask, parent, rank, w, h, npx, L,
                                 det->lab_area, det->lab_stride, det->flow, det->imu, det->det, det->max_det));
        MAVD_LAUNCHED();
        MAVD_CUDA(launch_chained(pdl_next(H), det_final_kernel, ceil_div(n * det->max_det, 128), 128, 0, s, det->det,
                                 n * det->max_det));
        MAVD_LAUNCHED();
    }
    return MAVD_OK;
}

// d_labels: the caller's label image (also used as the union-find array), or NULL when only the
// component count / boxes are wanted (the handle's scratch then holds the union-find array).
// list_ready: the producer of the mask already appended its occupied units (ccl_list_reset before it ran).
// det (nullable): also the detection table of every frame (DetArgs, common.cuh).
int ccl_run(mavd_handle H, const uint8_t* d_mask, int n, int32_t* d_labels, int32_t* d_boxes, size_t boxes_stride,
            int max_boxes, int32_t* d_n_labels, size_t nlabels_stride, cudaStream_t s, bool list_ready, const DetArgs* det) {
    ProfScope ps(&H->prof, MAVD_PROF_CCL, s);
    const int w = H->cfg.width;
    int* parent = d_labels ? d_labels : H->d_labels;
    const bool vec4 = (w % 4 == 0) && ((reinterpret_cast<uintptr_t>(d_mask) & 3) == 0);
    if (vec4) return ccl_launch<4>(H, d_mask, n, parent, d_labels, d_boxes, boxes_stride, max_boxes, d_n_labels, nlabels_stride, s, list_ready, det);
    return ccl_launch<1>(H, d_mask, n, parent, d_labels, d_boxes, boxes_stride, max_boxes, d_n_labels, nlabels_stride, s, list_ready, det);
}

}  // namespace mavd
