// Sparse feature path (sm_100a): cv2.goodFeaturesToTrack (Shi-Tomasi corners) and cv2.calcOpticalFlowPyrLK (pyramidal
// Lucas-Kanade), bit for bit where cv2's arithmetic is fixed-order (oracle/lk_np.py states what cv2 4.13 computes).
//
// Corners, per chunk of frames:
//   gftt_cov_kernel     Sobel (cv2's float32 rounding, fused multiply-adds where cv2's vector loop uses them) and the
//                       products dx*dx, dx*dy, dy*dy
//   gftt_rows_kernel    one thread per row: cv2's float64 running row sum of the block (direct sums for sizes 3, 5)
//   gftt_cols_kernel    one thread per column: cv2's float64 running column sum, lambda, the per-frame masked maximum
//   gftt_cand_kernel    quality threshold (float32), 3x3 local maximum, mask: appends (value, position) keys
//   gftt_sort_kernel    one CTA per frame: bitonic sort of the keys, descending (ties: later raster position first)
//   gftt_select_kernel  one warp per frame: greedy minimum-distance selection in rank order, 32 candidates at a time
//                       against a cell grid of accepted corners, conflicts inside the 32 resolved by ballot
// Tracker:
//   lk_pyr_down_kernel  cv2.pyrDown levels of every frame (exact integer arithmetic)
//   lk_scharr_kernel    int16 Scharr derivatives of every prev frame's levels
//   lk_track_kernel     one warp per point, all levels: the prev window (samples and derivatives) is staged in shared
//                       memory once per level, each iteration then resamples only the next frame
// The gradient matrix and mismatch vector are summed exactly in int64 (cv2 sums them in float32 in its SIMD lane order),
// so every point's result depends on its own inputs alone.  No kernel here is chained (plain launches only).
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace mavd {

namespace {

constexpr int kGfttChunk = 16;     // frames whose corner workspace is live at once
constexpr int kSobelVecCols = 32;  // cv2 4.13's u8 -> f32 row filter: fused multiply-adds in its vector loop
constexpr int kLkWarps = 4;        // points per tracker CTA

__device__ __forceinline__ int refl101(int p, int n) {
    if (n == 1) return 0;
    while ((unsigned)p >= (unsigned)n) p = p < 0 ? -p : 2 * n - 2 - p;
    return p;
}

// float -> uint32 with the same order (positive and negative values)
__device__ __forceinline__ uint32_t ord_f32(float v) {
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unord_f32(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

// ---------------------------------------------------------------------------------------------------------------------
// corner response

__global__ void gftt_cov_kernel(const uint8_t* __restrict__ frames, int W, int H, int bs, float3* __restrict__ cov) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const uint8_t* img = frames + (size_t)blockIdx.z * W * H;
    const float k1 = (float)(1.0 / (4.0 * bs * 255.0));
    const float k0 = __fmul_rn(2.f, k1);
    const int xm = refl101(x - 1, W), xp = refl101(x + 1, W);
    const int ym = refl101(y - 1, H), yp = refl101(y + 1, H);
    const uint8_t* r0 = img + (size_t)ym * W;
    const uint8_t* r1 = img + (size_t)y * W;
    const uint8_t* r2 = img + (size_t)yp * W;
    const int d0 = (int)r0[xp] - r0[xm], d1 = (int)r1[xp] - r1[xm], d2 = (int)r2[xp] - r2[xm];
    const float dx = __fmaf_rn((float)(d0 + d2), k1, __fmul_rn((float)d1, k0));
    float rowv[2];
    const bool fused = x < (W / kSobelVecCols) * kSobelVecCols;
    const uint8_t* rr[2] = {r0, r2};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float c0 = rr[i][xm], c1 = rr[i][x], c2 = rr[i][xp];
        rowv[i] = fused ? __fmaf_rn(c2, k1, __fmaf_rn(c1, k0, __fmul_rn(c0, k1)))
                        : __fadd_rn(__fadd_rn(__fmul_rn(c0, k1), __fmul_rn(c1, k0)), __fmul_rn(c2, k1));
    }
    const float dy = __fsub_rn(rowv[1], rowv[0]);
    cov[((size_t)blockIdx.z * H + y) * W + x] = make_float3(__fmul_rn(dx, dx), __fmul_rn(dx, dy), __fmul_rn(dy, dy));
}

__global__ void gftt_rows_kernel(const float3* __restrict__ cov, int W, int H, int bs, double* __restrict__ rows) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= H) return;
    const float3* c = cov + ((size_t)blockIdx.y * H + y) * W;
    double* out = rows + ((size_t)blockIdx.y * H + y) * W * 3;
    const int a = bs / 2;
    auto S = [&](int xp) { return c[refl101(xp - a, W)]; };   // xp: index into the row padded by the anchor
    if (bs == 3 || bs == 5) {
        for (int x = 0; x < W; ++x) {
            float3 v = S(x);
            double s0 = v.x, s1 = v.y, s2 = v.z;
            for (int i = 1; i < bs; ++i) {
                v = S(x + i);
                s0 = __dadd_rn(s0, (double)v.x); s1 = __dadd_rn(s1, (double)v.y); s2 = __dadd_rn(s2, (double)v.z);
            }
            out[3 * x] = s0; out[3 * x + 1] = s1; out[3 * x + 2] = s2;
        }
        return;
    }
    double s0 = 0, s1 = 0, s2 = 0;
    for (int i = 0; i < bs; ++i) {
        const float3 v = S(i);
        s0 = __dadd_rn(s0, (double)v.x); s1 = __dadd_rn(s1, (double)v.y); s2 = __dadd_rn(s2, (double)v.z);
    }
    out[0] = s0; out[1] = s1; out[2] = s2;
    for (int x = 1; x < W; ++x) {
        const float3 n = S(x + bs - 1), o = S(x - 1);
        s0 = __dadd_rn(s0, __dsub_rn((double)n.x, (double)o.x));
        s1 = __dadd_rn(s1, __dsub_rn((double)n.y, (double)o.y));
        s2 = __dadd_rn(s2, __dsub_rn((double)n.z, (double)o.z));
        out[3 * x] = s0; out[3 * x + 1] = s1; out[3 * x + 2] = s2;
    }
}

__global__ void gftt_cols_kernel(const double* __restrict__ rows, int W, int H, int bs, float* __restrict__ eig,
                                 const uint8_t* __restrict__ mask, int64_t mask_stride, uint32_t* __restrict__ maxv) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int f = blockIdx.y;
    uint32_t best = 0;
    if (x < W) {
        const double* R = rows + (size_t)f * H * W * 3 + 3 * x;
        float* E = eig + (size_t)f * H * W + x;
        const uint8_t* M = mask ? mask + (size_t)f * mask_stride + x : nullptr;
        const int a = bs / 2;
        auto row = [&](int yp) { return R + (size_t)refl101(yp - a, H) * W * 3; };
        double q0 = 0, q1 = 0, q2 = 0;
        for (int i = 0; i < bs - 1; ++i) {
            const double* r = row(i);
            q0 = __dadd_rn(q0, r[0]); q1 = __dadd_rn(q1, r[1]); q2 = __dadd_rn(q2, r[2]);
        }
        for (int y = 0; y < H; ++y) {
            const double* p = row(y + bs - 1);
            const double* m = row(y);
            const double s0 = __dadd_rn(q0, p[0]), s1 = __dadd_rn(q1, p[1]), s2 = __dadd_rn(q2, p[2]);
            q0 = __dsub_rn(s0, m[0]); q1 = __dsub_rn(s1, m[1]); q2 = __dsub_rn(s2, m[2]);
            const float ca = __fmul_rn(__double2float_rn(s0), 0.5f);
            const float cb = __double2float_rn(s1);
            const float cc = __fmul_rn(__double2float_rn(s2), 0.5f);
            const float t = __fsub_rn(ca, cc);
            const float lam = __fsub_rn(__fadd_rn(ca, cc), __fsqrt_rn(__fadd_rn(__fmul_rn(cb, cb), __fmul_rn(t, t))));
            E[(size_t)y * W] = lam;
            if (!M || M[(size_t)y * W]) best = max(best, ord_f32(lam));
        }
    }
    for (int o = 16; o; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0 && best) atomicMax(maxv + f, best);
}

__global__ void gftt_cand_kernel(const float* __restrict__ eig, int W, int H, const uint8_t* __restrict__ mask,
                                 int64_t mask_stride, const uint32_t* __restrict__ maxv, double quality,
                                 unsigned long long* __restrict__ keys, size_t key_cap, int* __restrict__ n_cand) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x + 1, y = blockIdx.y + 1, f = blockIdx.z;
    if (x > W - 2 || y > H - 2) return;
    const float* E = eig + (size_t)f * H * W;
    const uint32_t mo = maxv[f];
    const double mv = mo ? (double)unord_f32(mo) : 0.0;   // no pixel under the mask: cv2's maximum is 0
    const float thr = __double2float_rn(__dmul_rn(mv, quality));
    auto T = [&](int xx, int yy) { const float v = E[(size_t)yy * W + xx]; return v > thr ? v : 0.f; };
    const float v = T(x, y);
    if (v == 0.f) return;
    if (mask && !mask[(size_t)f * mask_stride + (size_t)y * W + x]) return;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx)
            if (T(x + dx, y + dy) > v) return;
    const int k = atomicAdd(n_cand + f, 1);
    keys[(size_t)f * key_cap + k] = ((unsigned long long)ord_f32(v) << 32) | (unsigned)(y * W + x);
}

// bitonic sort, descending, of one frame's keys (padded with zero keys, which no candidate has)
__global__ void __launch_bounds__(1024) gftt_sort_kernel(unsigned long long* __restrict__ keys, size_t key_cap,
                                                        const int* __restrict__ n_cand) {
    unsigned long long* K = keys + (size_t)blockIdx.x * key_cap;
    const int n = n_cand[blockIdx.x];
    if (n < 2) return;
    int N = 2;
    while (N < n) N <<= 1;
    for (int i = n + threadIdx.x; i < N; i += blockDim.x) K[i] = 0ull;
    __syncthreads();
    for (int k = 2; k <= N; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < N; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long a = K[i], b = K[l];
                    const bool desc = (i & k) == 0;
                    if (desc ? a < b : a > b) { K[i] = b; K[l] = a; }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void gftt_select_kernel(const unsigned long long* __restrict__ keys, size_t key_cap,
                                   const int* __restrict__ n_cand, int W, int H, double min_distance, int max_corners,
                                   int* __restrict__ grid, size_t grid_cap, float2* __restrict__ corners,
                                   int32_t* __restrict__ count) {
    const int f = blockIdx.x, lane = threadIdx.x;
    const unsigned long long* K = keys + (size_t)f * key_cap;
    const int n = n_cand[f];
    float2* out = corners ? corners + (size_t)f * max_corners : nullptr;
    int accepted = 0;
    if (!(min_distance > 1.0)) {   // distinct pixels are at least 1 apart: every candidate is kept
        for (int r = lane; r < min(n, max_corners); r += 32) {
            const unsigned p = (unsigned)K[r];
            out[r] = make_float2((float)(p % W), (float)(p / W));
        }
        accepted = n;
    } else {
        // cells of side ceil(min_distance) >= 2: a cell holds at most 4 accepted corners (one per quadrant), and a
        // corner closer than min_distance lies in one of the 3 x 3 cells around the candidate's
        const int c = (int)ceil(min_distance);
        const int gw = (W + c - 1) / c, gh = (H + c - 1) / c;
        int* G = grid + (size_t)f * grid_cap;
        const double md2 = min_distance * min_distance;
        const unsigned lt = (1u << lane) - 1u;
        for (int base = 0; base < n; base += 32) {
            const int r = base + lane;
            const bool valid = r < n;
            const unsigned p = valid ? (unsigned)K[r] : 0u;
            const int x = (int)(p % W), y = (int)(p / W);
            bool ok = valid;
            if (ok) {
                const int cx = x / c, cy = y / c;
                for (int gy = max(cy - 1, 0); ok && gy <= min(cy + 1, gh - 1); ++gy)
                    for (int gx = max(cx - 1, 0); ok && gx <= min(cx + 1, gw - 1); ++gx)
                        for (int s = 0; s < 4; ++s) {
                            const int v = G[((size_t)gy * gw + gx) * 4 + s];
                            if (!v) break;
                            const float ddx = (float)(x - (int)((unsigned)(v - 1) % W));
                            const float ddy = (float)(y - (int)((unsigned)(v - 1) / W));
                            if ((double)__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)) < md2) { ok = false; break; }
                        }
            }
            unsigned conf = 0;
            for (int j = 0; j < 32; ++j) {
                const int xj = __shfl_sync(0xffffffffu, x, j), yj = __shfl_sync(0xffffffffu, y, j);
                const float ddx = (float)(x - xj), ddy = (float)(y - yj);
                if (j < lane && (double)__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)) < md2) conf |= 1u << j;
            }
            const unsigned okm = __ballot_sync(0xffffffffu, ok);
            unsigned acc = 0;
            for (int j = 0; j < 32; ++j) {
                const unsigned cj = __shfl_sync(0xffffffffu, conf, j);
                if (((okm >> j) & 1u) && !(cj & acc)) acc |= 1u << j;
            }
            if ((acc >> lane) & 1u) {
                const int rank = accepted + __popc(acc & lt);
                if (rank < max_corners) out[rank] = make_float2((float)x, (float)y);
                int* cell = G + ((size_t)(y / c) * gw + x / c) * 4;
                for (int s = 0; s < 4; ++s)
                    if (atomicCAS(cell + s, 0, (int)p + 1) == 0) break;
            }
            accepted += __popc(acc);
            __syncwarp();
        }
    }
    for (int r = min(accepted, max_corners) + lane; r < max_corners; r += 32) out[r] = make_float2(0.f, 0.f);
    if (lane == 0) count[f] = accepted;
}

// ---------------------------------------------------------------------------------------------------------------------
// pyramidal Lucas-Kanade

struct LkGeom {
    int levels;                       // levels used (0 .. levels - 1)
    int w[MAVD_LK_MAX_LEVEL + 1], h[MAVD_LK_MAX_LEVEL + 1];
    size_t off[MAVD_LK_MAX_LEVEL + 1];    // byte offset of level l >= 1 inside a frame's pyramid block
    size_t doff[MAVD_LK_MAX_LEVEL + 1];   // element offset of level l inside a frame's derivative block
    size_t pyr_frame, der_frame;          // per-frame block sizes (bytes, short2 elements)
};

__device__ __forceinline__ const uint8_t* lk_level(const uint8_t* frames, const uint8_t* pyr, const LkGeom& g, int f,
                                                   int l) {
    return l == 0 ? frames + (size_t)f * g.w[0] * g.h[0] : pyr + (size_t)f * g.pyr_frame + g.off[l];
}

__global__ void lk_pyr_down_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ pyr, LkGeom g, int l) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    const int w = g.w[l], sw = g.w[l - 1], sh = g.h[l - 1];
    if (x >= w) return;
    const uint8_t* src = lk_level(frames, pyr, g, f, l - 1);
    const int k[5] = {1, 4, 6, 4, 1};
    int xs[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) xs[i] = refl101(2 * x + i - 2, sw);
    int tot = 0;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const uint8_t* r = src + (size_t)refl101(2 * y + j - 2, sh) * sw;
        int s = 0;
#pragma unroll
        for (int i = 0; i < 5; ++i) s += k[i] * r[xs[i]];
        tot += k[j] * s;
    }
    pyr[(size_t)f * g.pyr_frame + g.off[l] + (size_t)y * w + x] = (uint8_t)((tot + 128) >> 8);
}

__global__ void lk_scharr_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ pyr,
                                 short2* __restrict__ der, LkGeom g, int l, int pair_stride) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z * pair_stride;
    const int w = g.w[l], h = g.h[l];
    if (x >= w) return;
    const uint8_t* img = lk_level(frames, pyr, g, f, l);
    const uint8_t* r0 = img + (size_t)refl101(y - 1, h) * w;
    const uint8_t* r1 = img + (size_t)y * w;
    const uint8_t* r2 = img + (size_t)refl101(y + 1, h) * w;
    int t0[3], t1[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int xx = refl101(x + i - 1, w);
        t0[i] = (r0[xx] + r2[xx]) * 3 + r1[xx] * 10;
        t1[i] = r2[xx] - r0[xx];
    }
    der[(size_t)f * g.der_frame + g.doff[l] + (size_t)y * w + x] =
        make_short2((short)(t0[2] - t0[0]), (short)((t1[2] + t1[0]) * 3 + t1[1] * 10));
}

struct LkArgs {
    int win_w, win_h, iters, flags;
    double eps2;
    float min_eig;
    int pair_stride, n_points;
};

__device__ __forceinline__ long long warp_sum64(long long v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void lk_weights(float a, float b, int& w00, int& w01, int& w10, int& w11) {
    const float s = 16384.f;
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), __fsub_rn(1.f, b)), s));
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, __fsub_rn(1.f, b)), s));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), b), s));
    w11 = 16384 - w00 - w01 - w10;
}

__global__ void __launch_bounds__(kLkWarps * 32) lk_track_kernel(
    const uint8_t* __restrict__ frames, const uint8_t* __restrict__ pyr, const short2* __restrict__ der, LkGeom g,
    LkArgs A, const float2* __restrict__ prev_pts, const int32_t* __restrict__ n_pts, float2* __restrict__ next_pts,
    uint8_t* __restrict__ status, float* __restrict__ err) {
    extern __shared__ short lk_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int pair = blockIdx.y;
    const int i = blockIdx.x * kLkWarps + warp;
    if (i >= A.n_points) return;
    const size_t o = (size_t)pair * A.n_points + i;
    const int cnt = n_pts ? min(max(n_pts[pair], 0), A.n_points) : A.n_points;
    const float2 p = prev_pts[o];
    if (i >= cnt || !(isfinite(p.x) && isfinite(p.y))) {
        if (lane == 0) {
            next_pts[o] = i >= cnt ? make_float2(0.f, 0.f) : p;
            status[o] = 0;
            err[o] = 0.f;
        }
        return;
    }
    const int ww = A.win_w, wh = A.win_h, area = ww * wh;
    short* sI = lk_smem + (size_t)warp * area * 3;
    short* sX = sI + area;
    short* sY = sX + area;
    const float hwx = __fmul_rn((float)(ww - 1), 0.5f), hwy = __fmul_rn((float)(wh - 1), 0.5f);
    const float FLT_SCALE = 1.f / (1 << 20);
    const int fp = pair * A.pair_stride, fn = fp + 1;
    uint8_t st = 1;
    float e = 0.f;
    float nx = 0.f, ny = 0.f;
    const int L = g.levels - 1;
    for (int l = L; l >= 0; --l) {
        __syncwarp();
        const int w = g.w[l], h = g.h[l];
        const uint8_t* I = lk_level(frames, pyr, g, fp, l);
        const uint8_t* J = lk_level(frames, pyr, g, fn, l);
        const short2* D = der + (size_t)fp * g.der_frame + g.doff[l];
        const float sc = (float)(1.0 / (1 << l));
        float px = __fmul_rn(p.x, sc), py = __fmul_rn(p.y, sc);
        if (l == L) { nx = px; ny = py; } else { nx = __fmul_rn(nx, 2.f); ny = __fmul_rn(ny, 2.f); }
        px = __fsub_rn(px, hwx); py = __fsub_rn(py, hwy);
        const int ipx = (int)floorf(px), ipy = (int)floorf(py);
        if (ipx < -ww || ipx >= w || ipy < -wh || ipy >= h) {
            if (l == 0) { st = 0; e = 0.f; }
            continue;
        }
        int w00, w01, w10, w11;
        lk_weights(__fsub_rn(px, (float)ipx), __fsub_rn(py, (float)ipy), w00, w01, w10, w11);
        long long a11 = 0, a12 = 0, a22 = 0;
        for (int k = lane; k < area; k += 32) {
            const int wy = k / ww, wx = k - wy * ww;
            const int x0 = ipx + wx, y0 = ipy + wy;
            const int rx0 = refl101(x0, w), rx1 = refl101(x0 + 1, w);
            const uint8_t* r0 = I + (size_t)refl101(y0, h) * w;
            const uint8_t* r1 = I + (size_t)refl101(y0 + 1, h) * w;
            const int iv = (r0[rx0] * w00 + r0[rx1] * w01 + r1[rx0] * w10 + r1[rx1] * w11 + (1 << 8)) >> 9;
            short2 d[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int xx = x0 + (q & 1), yy = y0 + (q >> 1);
                d[q] = (xx >= 0 && xx < w && yy >= 0 && yy < h) ? D[(size_t)yy * w + xx] : make_short2(0, 0);
            }
            const int ix = (d[0].x * w00 + d[1].x * w01 + d[2].x * w10 + d[3].x * w11 + (1 << 13)) >> 14;
            const int iy = (d[0].y * w00 + d[1].y * w01 + d[2].y * w10 + d[3].y * w11 + (1 << 13)) >> 14;
            sI[k] = (short)iv; sX[k] = (short)ix; sY[k] = (short)iy;
            a11 += (long long)ix * ix; a12 += (long long)ix * iy; a22 += (long long)iy * iy;
        }
        a11 = warp_sum64(a11); a12 = warp_sum64(a12); a22 = warp_sum64(a22);
        __syncwarp();
        const float A11 = __fmul_rn(__ll2float_rn(a11), FLT_SCALE);
        const float A12 = __fmul_rn(__ll2float_rn(a12), FLT_SCALE);
        const float A22 = __fmul_rn(__ll2float_rn(a22), FLT_SCALE);
        const float Dt = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float t = __fsub_rn(A11, A22);
        const float min_eig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), __fsqrt_rn(__fadd_rn(__fmul_rn(t, t),
                                                   __fmul_rn(__fmul_rn(4.f, A12), A12)))), (float)(2 * area));
        if (A.flags & MAVD_LK_GET_MIN_EIGENVALS) e = min_eig;
        if (min_eig < A.min_eig || Dt < 1.1920928955078125e-7f) {
            if (l == 0) st = 0;
            continue;
        }
        const float Dinv = __fdiv_rn(1.f, Dt);
        float cx = __fsub_rn(nx, hwx), cy = __fsub_rn(ny, hwy);
        float pdx = 0.f, pdy = 0.f;
        for (int j = 0; j < A.iters; ++j) {
            const int inx = (int)floorf(cx), iny = (int)floorf(cy);
            if (inx < -ww || inx >= w || iny < -wh || iny >= h) {
                if (l == 0) st = 0;
                break;
            }
            lk_weights(__fsub_rn(cx, (float)inx), __fsub_rn(cy, (float)iny), w00, w01, w10, w11);
            long long b1 = 0, b2 = 0;
            for (int k = lane; k < area; k += 32) {
                const int wy = k / ww, wx = k - wy * ww;
                const int x0 = inx + wx, y0 = iny + wy;
                const int rx0 = refl101(x0, w), rx1 = refl101(x0 + 1, w);
                const uint8_t* r0 = J + (size_t)refl101(y0, h) * w;
                const uint8_t* r1 = J + (size_t)refl101(y0 + 1, h) * w;
                const int diff = ((r0[rx0] * w00 + r0[rx1] * w01 + r1[rx0] * w10 + r1[rx1] * w11 + (1 << 8)) >> 9) - sI[k];
                b1 += (long long)diff * sX[k];
                b2 += (long long)diff * sY[k];
            }
            b1 = warp_sum64(b1); b2 = warp_sum64(b2);
            const float B1 = __fmul_rn(__ll2float_rn(b1), FLT_SCALE), B2 = __fmul_rn(__ll2float_rn(b2), FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, B2), __fmul_rn(A22, B1)), Dinv);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, B1), __fmul_rn(A11, B2)), Dinv);
            cx = __fadd_rn(cx, dx); cy = __fadd_rn(cy, dy);
            nx = __fadd_rn(cx, hwx); ny = __fadd_rn(cy, hwy);
            if (__dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= A.eps2) break;
            if (j > 0 && fabsf(__fadd_rn(dx, pdx)) < 0.01 && fabsf(__fadd_rn(dy, pdy)) < 0.01) {
                nx = __fsub_rn(nx, __fmul_rn(dx, 0.5f));
                ny = __fsub_rn(ny, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx; pdy = dy;
        }
        if (l == 0 && st && !(A.flags & MAVD_LK_GET_MIN_EIGENVALS)) {
            const float qx = __fsub_rn(nx, hwx), qy = __fsub_rn(ny, hwy);
            const int iqx = (int)floorf(qx), iqy = (int)floorf(qy);
            if (iqx < -ww || iqx >= w || iqy < -wh || iqy >= h) {
                st = 0;
                continue;
            }
            lk_weights(__fsub_rn(qx, (float)iqx), __fsub_rn(qy, (float)iqy), w00, w01, w10, w11);
            long long s = 0;
            for (int k = lane; k < area; k += 32) {
                const int wy = k / ww, wx = k - wy * ww;
                const int x0 = iqx + wx, y0 = iqy + wy;
                const int rx0 = refl101(x0, w), rx1 = refl101(x0 + 1, w);
                const uint8_t* r0 = J + (size_t)refl101(y0, h) * w;
                const uint8_t* r1 = J + (size_t)refl101(y0 + 1, h) * w;
                const int diff = ((r0[rx0] * w00 + r0[rx1] * w01 + r1[rx0] * w10 + r1[rx1] * w11 + (1 << 8)) >> 9) - sI[k];
                s += diff < 0 ? -diff : diff;
            }
            s = warp_sum64(s);
            e = __fdiv_rn(__ll2float_rn(s), (float)(32 * area));
        }
        __syncwarp();
    }
    if (lane == 0) {
        next_pts[o] = make_float2(nx, ny);
        status[o] = st;
        err[o] = e;
    }
}

}  // namespace

// workspace sizes of the sparse path (allocated on first use by api.cu)
size_t gftt_key_cap(int W, int H) {
    size_t n = (size_t)max(W - 2, 1) * (size_t)max(H - 2, 1), c = 2;
    while (c < n) c <<= 1;
    return c;
}
size_t gftt_grid_cap(int W, int H) { return (size_t)((W + 1) / 2) * ((H + 1) / 2) * 4; }
int gftt_chunk() { return kGfttChunk; }

int gftt_run(mavd_handle h, const GfttWork& ws, const uint8_t* d_frames, int n, const mavd_gftt_params& p,
             const uint8_t* d_mask, int64_t mask_stride, float* d_corners, int32_t* d_count, float* d_eig,
             cudaStream_t s) {
    const int W = h->cfg.width, H = h->cfg.height;
    const size_t npx = (size_t)W * H;
    const size_t kcap = gftt_key_cap(W, H), gcap = gftt_grid_cap(W, H);
    const bool grid = p.min_distance > 1.0;
    for (int f0 = 0; f0 < n; f0 += kGfttChunk) {
        const int g = min(kGfttChunk, n - f0);
        const uint8_t* fr = d_frames + (size_t)f0 * npx;
        const uint8_t* mk = d_mask ? d_mask + (size_t)f0 * mask_stride : nullptr;
        float* eig = d_eig ? d_eig + (size_t)f0 * npx : ws.eig;
        MAVD_CUDA(cudaMemsetAsync(ws.maxv, 0, sizeof(uint32_t) * g, s));
        MAVD_CUDA(cudaMemsetAsync(ws.n_cand, 0, sizeof(int) * g, s));
        gftt_cov_kernel<<<dim3(ceil_div(W, 128), H, g), 128, 0, s>>>(fr, W, H, p.block_size, ws.cov);
        MAVD_LAUNCHED();
        gftt_rows_kernel<<<dim3(ceil_div(H, 64), g), 64, 0, s>>>(ws.cov, W, H, p.block_size, ws.rows);
        MAVD_LAUNCHED();
        gftt_cols_kernel<<<dim3(ceil_div(W, 64), g), 64, 0, s>>>(ws.rows, W, H, p.block_size, eig, mk, mask_stride,
                                                                 ws.maxv);
        MAVD_LAUNCHED();
        if (W >= 3 && H >= 3) {
            gftt_cand_kernel<<<dim3(ceil_div(W - 2, 128), H - 2, g), 128, 0, s>>>(eig, W, H, mk, mask_stride, ws.maxv,
                                                                                   p.quality_level, ws.keys, kcap,
                                                                                   ws.n_cand);
            MAVD_LAUNCHED();
        }
        gftt_sort_kernel<<<g, 1024, 0, s>>>(ws.keys, kcap, ws.n_cand);
        MAVD_LAUNCHED();
        if (grid) MAVD_CUDA(cudaMemsetAsync(ws.grid, 0, sizeof(int) * gcap * g, s));
        gftt_select_kernel<<<g, 32, 0, s>>>(ws.keys, kcap, ws.n_cand, W, H, p.min_distance, p.max_corners, ws.grid, gcap,
                                            d_corners ? (float2*)d_corners + (size_t)f0 * p.max_corners : nullptr,
                                            d_count + f0);
        MAVD_LAUNCHED();
    }
    return MAVD_OK;
}

int lk_levels(int W, int H, int win_w, int win_h, int max_level) {
    int w = W, hh = H;
    for (int l = 0; l <= max_level; ++l) {
        w = (w + 1) / 2; hh = (hh + 1) / 2;
        if (w <= win_w || hh <= win_h) return l + 1;
    }
    return max_level + 1;
}

static LkGeom lk_geom(int W, int H, int levels) {
    LkGeom g;
    memset(&g, 0, sizeof(g));
    g.levels = levels;
    g.w[0] = W; g.h[0] = H;
    size_t off = 0, doff = (size_t)W * H;
    for (int l = 1; l <= MAVD_LK_MAX_LEVEL; ++l) {
        g.w[l] = (g.w[l - 1] + 1) / 2; g.h[l] = (g.h[l - 1] + 1) / 2;
        g.off[l] = off; g.doff[l] = doff;
        off += (size_t)g.w[l] * g.h[l];
        doff += (size_t)g.w[l] * g.h[l];
    }
    g.pyr_frame = off;
    g.der_frame = doff;
    return g;
}
size_t lk_pyr_frame_bytes(int W, int H) { return lk_geom(W, H, 1).pyr_frame; }
size_t lk_der_frame_elems(int W, int H) { return lk_geom(W, H, 1).der_frame; }

int lk_run(mavd_handle h, uint8_t* pyr, short2* der, const uint8_t* d_frames, int n_pairs, int pair_stride,
           const mavd_lk_params& p, const float* d_prev, int n_points, const int32_t* d_n_points, float* d_next,
           uint8_t* d_status, float* d_err, cudaStream_t s) {
    const int W = h->cfg.width, H = h->cfg.height;
    const LkGeom g = lk_geom(W, H, lk_levels(W, H, p.win_w, p.win_h, p.max_level));
    const int n_frames = (n_pairs - 1) * pair_stride + 2;
    for (int l = 1; l < g.levels; ++l) {
        lk_pyr_down_kernel<<<dim3(ceil_div(g.w[l], 128), g.h[l], n_frames), 128, 0, s>>>(d_frames, pyr, g, l);
        MAVD_LAUNCHED();
    }
    for (int l = 0; l < g.levels; ++l) {
        lk_scharr_kernel<<<dim3(ceil_div(g.w[l], 128), g.h[l], n_pairs), 128, 0, s>>>(d_frames, pyr, der, g, l,
                                                                                         pair_stride);
        MAVD_LAUNCHED();
    }
    LkArgs a;
    a.win_w = p.win_w; a.win_h = p.win_h; a.flags = p.flags;
    a.iters = (p.criteria_type & MAVD_TERM_COUNT) ? min(max(p.criteria_count, 0), 100) : 30;
    const double eps = (p.criteria_type & MAVD_TERM_EPS) ? fmin(fmax(p.criteria_eps, 0.0), 10.0) : 0.01;
    a.eps2 = eps * eps;
    a.min_eig = (float)p.min_eig_threshold;
    a.pair_stride = pair_stride;
    a.n_points = n_points;
    const size_t smem = (size_t)kLkWarps * p.win_w * p.win_h * 3 * sizeof(short);
    // the opt-in is made once per device, so it is made for the largest window
    MAVD_CUDA(ensure_dynamic_smem<lk_track_kernel>((size_t)kLkWarps * 63 * 63 * 3 * sizeof(short)));
    lk_track_kernel<<<dim3(ceil_div(n_points, kLkWarps), n_pairs), kLkWarps * 32, smem, s>>>(
        d_frames, pyr, der, g, a, (const float2*)d_prev, d_n_points, (float2*)d_next, d_status, d_err);
    MAVD_LAUNCHED();
    return MAVD_OK;
}

}  // namespace mavd
