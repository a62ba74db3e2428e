// Farneback dense optical flow for sm_100a — the arithmetic of cv2.calcOpticalFlowFarneback as
// called at /root/reference/src/farneback.py:76-80 (SURVEY.md §8 a2-a7, Appendix A).
//
// HBM layout: every per-level field is PLANAR with a row pitch that is a multiple of 64 floats
// (256 B): image [frame][h][pitch]; R [frame][5][h][pitch]; M [pair][5][h][pitch] (ping-pong);
// flow [pair][h][pitch] float2.  64-wide tiles therefore never cross a row end and every tile row is
// 16-byte aligned (float4 / cp.async / TMA friendly).  Batch elements sit in grid.z, or lead the grid (grid.x, or
// interleaved into a 1-D grid) where the CTA order matters for L2 (consecutive pairs share an R plane).
//
// Kernels (algorithmic bytes per level pixel P, per SURVEY §8d):
//   pyr_vfirst / pyr_hsecond / pyr_hsecond_staged
//                             blur+resize from full-res u8 for all coarse levels, any pyr_scale (generic)
//   pyr_vsweep / pyr_hpass / pyr_hpass1
//                             the same for the exact power-of-two levels of a pyr_scale 0.5 pyramid: one sweep down the
//                             frame does the vertical passes of levels 1..4 (each u8 row converted once) and level
//                             1's horizontal pass; vectorised / streamed horizontal passes for the other levels
//   polyexp_tma_kernel        separable polynomial expansion, tile staged by one TMA box  4P -> 20P (level 0: 1P -> 20P)
//   polyexp_kernel            the same with per-thread loads (rows that are not 16-byte aligned)
//   matrices_init_kernel      flow upsample (x 1/pyr_scale) fused with UpdateMatrices   (8P' +) 40P -> 20P
//   iter_box_tma_kernel       box / Gaussian blur of M + 2x2 solve + UpdateMatrices, TMA-staged, window half-widths
//                             5..8 (winsize 10..17), 64x32 or 64x16 tiles                88P (28P for the last)
//   iter_kernel               the same for the other window sizes (generic staging); reference of the bit-equality tests
#include <math.h>

#include "common.cuh"

namespace mavd {

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int i, int n) {
    // BORDER_REFLECT_101:  ... c b | a b c ... y z | y x ...
    while (i < 0 || i >= n) {
        if (n == 1) return 0;
        i = (i < 0) ? -i : 2 * (n - 1) - i;
    }
    return i;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// ------------------------------------------------------------------------------------------------
// Pyramid: I_l = resize(GaussianBlur(f32(img), ksz, sigma), (w_l, h_l)), always from full resolution.
// Blur and bilinear resize are both linear and separable, so per axis they collapse into ONE filter of
// ksz+1 taps per output sample: c_j = (1-a) k_j + a k_{j-1} at source index i0 - r + j (REFLECT_101).
// Level 0 (sigma 0 -> [1/4 1/2 1/4], identity resize) is fused into the polynomial expansion's tile
// staging and never touches HBM.  All coarser levels share two launches:
//   pyr_vfirst   vertical filter straight from the u8 frame: thread = 4 adjacent columns (one 32-bit word per
//                tap row, coalesced, no staging) x one output row; the tap weight is warp-uniform;
//                writes tmp_l [h_l][Wp] float for every level
//   pyr_hsecond  horizontal filter on tmp_l: thread = one output pixel, x fastest
// Doing the vertical pass first shrinks the row count before the expensive direction: 4 full-rate
// instructions per u8 tap (byte permute, exact mantissa-trick convert, FMA) and no shared memory.
// ------------------------------------------------------------------------------------------------
struct PyrLevel {
    int w, h, pitch, taps;
    const int* xbase; const float* xtab;   // [w], [w][taps]
    const float* xtabT;                     // [taps][w]: the same weights, tap-major (pyr_hsecond_staged_kernel)
    int staged;                             // horizontal pass through shared memory (source stride >= 8, span fits)
    const int* ybase; const float* ytab;   // [h], [h][taps]
    float* tmp; float* img;
    size_t tmp_stride, img_stride;          // floats per frame
    // both passes run on a 3-D grid (tile column, row tile of any level, frame): no integer division per thread; the
    // levels share the y range ([row0, row0 + ceil(h / 4)) belongs to this level), blocks right of a narrow level exit
    int row0;                               // first row tile (4 rows) of this level in grid.y
    int htiles_x;                           // pyr_hsecond: 64-pixel tiles per row (pyr_vfirst: ceil(W / 256) for all)
};
struct PyrDesc {
    int n;
    PyrLevel lv[kMaxLevels];
};

// u8 -> float without a conversion instruction: byte k of v placed in the mantissa of 2^23, then - 2^23 (exact)
__device__ __forceinline__ float byte_to_float(uint32_t v, uint32_t selector) {
    return __uint_as_float(__byte_perm(v, 0x4B000000u, selector)) - 8388608.f;
}

__global__ void __launch_bounds__(256) pyr_vfirst_kernel(const uint8_t* __restrict__ frames, size_t frame_stride, int W,
                                                        int H, int Wp, int word_ok, const __grid_constant__ PyrDesc d) {
    pdl_entry();
    int l = 0;
    while (l + 1 < d.n && (int)blockIdx.y >= d.lv[l + 1].row0) ++l;
    const PyrLevel& L = d.lv[l];
    const int x = (blockIdx.x * 64 + (threadIdx.x & 63)) * 4, dy = (blockIdx.y - L.row0) * 4 + (threadIdx.x >> 6);
    if (x >= W || dy >= L.h) return;
    const uint8_t* src = frames + (size_t)blockIdx.z * frame_stride + x;
    const int base = __ldg(L.ybase + dy);
    const float* tab = L.ytab + dy * L.taps;
    const int taps = L.taps;
    const bool inside = base >= 0 && base + taps <= H;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    if (word_ok && x + 4 <= W && inside) {
        // interior: walk down the rows with a pointer, four taps (one float4 of weights) per step
        const uint8_t* q = src + (size_t)base * W;
        for (int j = 0; j < taps; j += 4) {          // taps is a multiple of 4 (zero padded)
            const float4 t = __ldg(reinterpret_cast<const float4*>(tab + j));
            const uint32_t v0 = __ldg(reinterpret_cast<const uint32_t*>(q));
            const uint32_t v1 = __ldg(reinterpret_cast<const uint32_t*>(q + W));
            const uint32_t v2 = __ldg(reinterpret_cast<const uint32_t*>(q + 2 * (size_t)W));
            const uint32_t v3 = __ldg(reinterpret_cast<const uint32_t*>(q + 3 * (size_t)W));
            q += 4 * (size_t)W;
            a0 += t.x * byte_to_float(v0, 0x7540u); a1 += t.x * byte_to_float(v0, 0x7541u);
            a2 += t.x * byte_to_float(v0, 0x7542u); a3 += t.x * byte_to_float(v0, 0x7543u);
            a0 += t.y * byte_to_float(v1, 0x7540u); a1 += t.y * byte_to_float(v1, 0x7541u);
            a2 += t.y * byte_to_float(v1, 0x7542u); a3 += t.y * byte_to_float(v1, 0x7543u);
            a0 += t.z * byte_to_float(v2, 0x7540u); a1 += t.z * byte_to_float(v2, 0x7541u);
            a2 += t.z * byte_to_float(v2, 0x7542u); a3 += t.z * byte_to_float(v2, 0x7543u);
            a0 += t.w * byte_to_float(v3, 0x7540u); a1 += t.w * byte_to_float(v3, 0x7541u);
            a2 += t.w * byte_to_float(v3, 0x7542u); a3 += t.w * byte_to_float(v3, 0x7543u);
        }
    } else if (word_ok && x + 4 <= W) {
        for (int j = 0; j < taps; ++j) {
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)reflect101(base + j, H) * W));
            const float t = __ldg(tab + j);
            a0 += t * byte_to_float(v, 0x7540u);
            a1 += t * byte_to_float(v, 0x7541u);
            a2 += t * byte_to_float(v, 0x7542u);
            a3 += t * byte_to_float(v, 0x7543u);
        }
    } else {
        const int nx = min(4, W - x);
        for (int j = 0; j < taps; ++j) {
            const uint8_t* q = src + (size_t)reflect101(base + j, H) * W;
            const float t = __ldg(tab + j);
            a0 += t * (float)q[0];
            if (nx > 1) a1 += t * (float)q[1];
            if (nx > 2) a2 += t * (float)q[2];
            if (nx > 3) a3 += t * (float)q[3];
        }
    }
    float* out = L.tmp + (size_t)blockIdx.z * L.tmp_stride + (size_t)dy * Wp + x;
    *reinterpret_cast<float4*>(out) = make_float4(a0, a1, a2, a3);   // Wp is a multiple of 4: the pad is never read
}

__global__ void __launch_bounds__(256) pyr_hsecond_kernel(int W, int Wp, int row_begin, const __grid_constant__ PyrDesc d) {
    pdl_entry();
    const int by = blockIdx.y + row_begin;
    int l = 0;
    while (l + 1 < d.n && by >= d.lv[l + 1].row0) ++l;
    const PyrLevel& L = d.lv[l];
    if ((int)blockIdx.x >= L.htiles_x || L.staged) return;
    const int dx = blockIdx.x * 64 + (threadIdx.x & 63), dy = (by - L.row0) * 4 + (threadIdx.x >> 6);
    if (dx >= L.w || dy >= L.h) return;
    const float* src = L.tmp + (size_t)blockIdx.z * L.tmp_stride + (size_t)dy * Wp;
    const int base = __ldg(L.xbase + dx);
    const float* tab = L.xtab + dx * L.taps;
    const int taps = L.taps;
    float acc = 0.f;
    if (base >= 0 && base + taps <= W) {
        for (int j = 0; j < taps; j += 4) {     // taps is a multiple of 4 (zero padded)
            const float4 t = __ldg(reinterpret_cast<const float4*>(tab + j));
            acc += t.x * src[base + j];
            acc += t.y * src[base + j + 1];
            acc += t.z * src[base + j + 2];
            acc += t.w * src[base + j + 3];
        }
    } else {
        for (int j = 0; j < taps; ++j) acc += __ldg(tab + j) * src[reflect101(base + j, W)];
    }
    L.img[(size_t)blockIdx.z * L.img_stride + (size_t)dy * L.pitch + dx] = acc;
}

// Horizontal pass of the coarse levels (source stride >= 8 floats between adjacent outputs).  Read directly, the 32
// lanes of a warp touch 8 .. 32 different 128-byte lines per tap; here the block first copies the source span of its
// 64 outputs x 4 rows into shared memory with coalesced loads, stored with one pad word per 32 (index e + e / 32) so
// that lanes a power-of-two stride apart fall into different banks, and reads the weights tap-major (coalesced).
// Same products, same order of accumulation as pyr_hsecond_kernel.
constexpr int PYR_SPAN_MAX = 2208;                               // source floats per row a block may stage
constexpr int PYR_SPAN_PAD = PYR_SPAN_MAX + PYR_SPAN_MAX / 32 + 3;

__global__ void __launch_bounds__(256) pyr_hsecond_staged_kernel(int W, int Wp, int row_begin,
                                                                const __grid_constant__ PyrDesc d) {
    pdl_entry();
    __shared__ float s_src[4][PYR_SPAN_PAD];
    const int by = blockIdx.y + row_begin;
    int l = 0;
    while (l + 1 < d.n && by >= d.lv[l + 1].row0) ++l;
    const PyrLevel& L = d.lv[l];
    if ((int)blockIdx.x >= L.htiles_x || !L.staged) return;
    const int i = threadIdx.x & 63, ry = threadIdx.x >> 6;
    const int dx0 = blockIdx.x * 64, dx = dx0 + i, dy = (by - L.row0) * 4 + ry;
    const int taps = L.taps;
    const int lo = __ldg(L.xbase + dx0), hi = __ldg(L.xbase + min(dx0 + 63, L.w - 1)) + taps;
    const int n = hi - lo;                                   // <= PYR_SPAN_MAX (checked on the host)
    if (dy < L.h) {
        const float* src = L.tmp + (size_t)blockIdx.z * L.tmp_stride + (size_t)dy * Wp;
        float* dst = s_src[ry];
        if (lo >= 0 && hi <= W) {
            for (int e = i; e < n; e += 64) dst[e + (e >> 5)] = src[lo + e];
        } else {
            for (int e = i; e < n; e += 64) dst[e + (e >> 5)] = src[reflect101(lo + e, W)];
        }
    }
    __syncthreads();
    if (dx >= L.w || dy >= L.h) return;
    const float* row = s_src[ry];
    const float* wt = L.xtabT + dx;
    const int b = __ldg(L.xbase + dx) - lo;
    const int w = L.w;
    float acc = 0.f;
    for (int j = 0; j < taps; j += 4) {     // taps is a multiple of 4 (zero padded)
        const int e = b + j;
        acc += __ldg(wt + (size_t)j * w) * row[e + (e >> 5)];
        acc += __ldg(wt + (size_t)(j + 1) * w) * row[(e + 1) + ((e + 1) >> 5)];
        acc += __ldg(wt + (size_t)(j + 2) * w) * row[(e + 2) + ((e + 2) >> 5)];
        acc += __ldg(wt + (size_t)(j + 3) * w) * row[(e + 3) + ((e + 3) >> 5)];
    }
    L.img[(size_t)blockIdx.z * L.img_stride + (size_t)dy * L.pitch + dx] = acc;
}

// ------------------------------------------------------------------------------------------------
// Exact power-of-two levels (pyr_scale 0.5, frame size divisible by 2^l; api.cu checks the tables): every output
// sample of level l has the SAME T = ksz + 1 weights and its window starts S = 2^l samples after its neighbour's,
// at S * d - NB.  The generic kernels above do not know that: they convert every u8 sample once per tap that uses it
// (2.5 times per level) and spend most of their instructions finding their level and their table rows.
//   pyr_vsweep   vertical pass of levels 1..NLV in ONE sweep down the frame: thread = 4 adjacent columns (one 32-bit
//                word per row, coalesced), each row is loaded and converted once and added to the <= 3 live output
//                rows of every level (polyphase decimation: the tap index of (row, live output) is a compile-time
//                constant, the weight a uniform-register operand of the FFMA); a finished output row is stored and its
//                accumulator starts the next one.  ~20 instead of ~50 instructions per source sample for three levels.
//   pyr_hpass    horizontal pass of level 1 or 2: thread = 4 adjacent outputs of one row, source span read as float4
//   pyr_hpass1   horizontal pass of levels 3..6 (windows of 20..160 samples, 8..64 apart): thread = one output, its
//                window streamed as float4 groups (the staged generic kernel spends 600 instructions per output on
//                copying spans into shared memory)
// Per output sample the products are accumulated in the same tap order with the same FMAs as in the generic kernels:
// the images are bit-identical (test_pyramid_sweep_equals_the_generic_kernels).
// ------------------------------------------------------------------------------------------------
struct HalfPyr {    // level l = 1..6: stride, taps, -(window start of output 0), live outputs per source row
    __host__ __device__ static constexpr int S(int l) { return 1 << l; }
    __host__ __device__ static constexpr int T(int l) { return l == 1 ? 4 : 10 << (l - 2); }        // 4 10 20 40 80 160
    __host__ __device__ static constexpr int NB(int l) { return l == 1 ? 1 : 3 << (l - 2); }        // 1 3 6 12 24 48
    __host__ __device__ static constexpr int K(int l) { return (T(l) + S(l) - 1) / S(l); }
};
constexpr int VS_MAXLV = 4, VS_MAXT = 40;      // levels one sweep takes; their taps
constexpr int HP_MAXLV = 6, HP_MAXT = 160;     // levels with a uniform horizontal pass; their taps
struct VSweepDesc {
    float* tmp[VS_MAXLV];
    size_t tmp_stride[VS_MAXLV];   // floats per frame
    int h[VS_MAXLV];
    float w[VS_MAXLV][VS_MAXT];
    int band_rows;                 // output rows of level NLV per band (grid.y)
    // H1: level 1's horizontal pass inside the sweep (its image instead of its tmp rows)
    float* img1; size_t img1_stride; int pitch1;
    float xw1[4];
};

// H1: the thread also filters the column left and the column right of its four (REFLECT_101 at the frame edge) for
// level 1, so that a finished level-1 row gets its horizontal pass (two outputs per thread, four taps) on the spot and
// goes to the level image: the 4 bytes per full-resolution column of tmp never make their round trip through HBM
// (270 MB written + 270 MB read per 65 frames of 1080p, what the sweep and pyr_hpass<1> were bound by).
template <int NLV, bool H1>
__global__ void __launch_bounds__(192) pyr_vsweep_kernel(const uint8_t* __restrict__ frames, size_t frame_stride, int W,
                                                        int H, int Wp, const __grid_constant__ VSweepDesc d) {
    pdl_entry();
    constexpr int U = 1 << NLV;      // source rows per unrolled step = stride of the coarsest swept level
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (x >= W) return;
    const uint8_t* src = frames + (size_t)blockIdx.z * frame_stride + x;
    const int D0 = blockIdx.y * d.band_rows, D1 = min(D0 + d.band_rows, d.h[NLV - 1]);
    float acc[NLV][3][4];
#pragma unroll
    for (int l = 0; l < NLV; ++l)
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[l][k][c] = 0.f;
    float e1[2][2] = {{0.f, 0.f}, {0.f, 0.f}};       // H1: level 1, [k][left / right neighbour column]
    // neighbour columns: byte 3 of the word on the left, byte 0 of the word on the right; at the frame edge the
    // reflected column is byte 1 / byte 2 of the thread's own word
    const int offl = x >= 4 ? -4 : 0, offr = x + 4 < W ? 4 : 0;
    const uint32_t sell = x >= 4 ? 0x7543u : 0x7541u, selr = x + 4 < W ? 0x7540u : 0x7542u;
    // the window of output D0 of level l starts at U * D0 - NB(l) >= U * (D0 - 1); that of output D1 - 1 ends before
    // U * (D1 + 2): steps q = D0 - 1 .. D1 + 1.  Outputs outside the band (their sums are incomplete) are not stored.
#pragma unroll 1
    for (int q = D0 - 1; q <= D1 + 1; ++q) {
        const int r0 = q * U;
        uint32_t wv[U], wl[H1 ? U : 1], wr[H1 ? U : 1];
        if (r0 >= 0 && r0 + U <= H) {
            const uint8_t* p = src + (size_t)r0 * W;
#pragma unroll
            for (int i = 0; i < U; ++i) {
                wv[i] = __ldg(reinterpret_cast<const uint32_t*>(p + (size_t)i * W));
                if (H1) {
                    wl[i] = __ldg(reinterpret_cast<const uint32_t*>(p + (size_t)i * W + offl));
                    wr[i] = __ldg(reinterpret_cast<const uint32_t*>(p + (size_t)i * W + offr));
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < U; ++i) {
                const uint8_t* p = src + (size_t)reflect101(r0 + i, H) * W;
                wv[i] = __ldg(reinterpret_cast<const uint32_t*>(p));
                if (H1) {
                    wl[i] = __ldg(reinterpret_cast<const uint32_t*>(p + offl));
                    wr[i] = __ldg(reinterpret_cast<const uint32_t*>(p + offr));
                }
            }
        }
#pragma unroll
        for (int i = 0; i < U; ++i) {
            const float v[4] = {byte_to_float(wv[i], 0x7540u), byte_to_float(wv[i], 0x7541u),
                                byte_to_float(wv[i], 0x7542u), byte_to_float(wv[i], 0x7543u)};
#pragma unroll
            for (int l = 1; l <= NLV; ++l) {
                const int S = HalfPyr::S(l), T = HalfPyr::T(l), NB = HalfPyr::NB(l), K = HalfPyr::K(l);
                const int ph = (i + NB) % S;                 // row r0 + i is tap ph + k S of the k-th newest output
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    if (k < K && ph + k * S < T) {
                        const float wt = d.w[l - 1][ph + k * S];
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[l - 1][k][c] = fmaf(wt, v[c], acc[l - 1][k][c]);
                        if (H1 && l == 1) {
                            e1[k][0] = fmaf(wt, byte_to_float(wl[i], sell), e1[k][0]);
                            e1[k][1] = fmaf(wt, byte_to_float(wr[i], selr), e1[k][1]);
                        }
                    }
                if (ph == S - 1) {
                    // the oldest live output is complete: index = newest - (K - 1)
                    const int dn = (U / S) * q + (i + NB) / S - (K - 1);
                    if (dn >= D0 * (U / S) && dn < min(D1 * (U / S), d.h[l - 1])) {
                        if (H1 && l == 1) {
                            // outputs x / 2 and x / 2 + 1 of the level-1 row: columns x - 1 .. x + 2 and x + 1 .. x + 4
                            const float c6[6] = {e1[K - 1][0], acc[0][K - 1][0], acc[0][K - 1][1], acc[0][K - 1][2],
                                                 acc[0][K - 1][3], e1[K - 1][1]};
                            float o0 = 0.f, o1 = 0.f;
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                o0 = fmaf(d.xw1[j], c6[j], o0);
                                o1 = fmaf(d.xw1[j], c6[2 + j], o1);
                            }
                            float* out = d.img1 + (size_t)blockIdx.z * d.img1_stride + (size_t)dn * d.pitch1 + (x >> 1);
                            *reinterpret_cast<float2*>(out) = make_float2(o0, o1);
                        } else {
                            float* out = d.tmp[l - 1] + (size_t)blockIdx.z * d.tmp_stride[l - 1] + (size_t)dn * Wp + x;
                            *reinterpret_cast<float4*>(out) = make_float4(acc[l - 1][K - 1][0], acc[l - 1][K - 1][1],
                                                                         acc[l - 1][K - 1][2], acc[l - 1][K - 1][3]);
                        }
                    }
                    if (H1 && l == 1) {
                        e1[1][0] = e1[0][0]; e1[1][1] = e1[0][1];
                        e1[0][0] = e1[0][1] = 0.f;
                    }
#pragma unroll
                    for (int k = 2; k >= 1; --k)
                        if (k < K) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) acc[l - 1][k][c] = acc[l - 1][k - 1][c];
                        }
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[l - 1][0][c] = 0.f;
                }
            }
        }
    }
}

struct HPassW { float w[HP_MAXT]; };

template <int LV>
__global__ void __launch_bounds__(128) pyr_hpass_kernel(const float* __restrict__ tmp, size_t tmp_stride, int W, int Wp,
                                                       int wl, float* __restrict__ img, size_t img_stride, int pitch,
                                                       const __grid_constant__ HPassW wts) {
    pdl_entry();
    constexpr int S = HalfPyr::S(LV), T = HalfPyr::T(LV), NB = HalfPyr::NB(LV);
    constexpr int OFF = (4 - NB % 4) % 4;               // the window of output x starts OFF floats into a 16-byte group
    constexpr int NV = (OFF + 3 * S + T + 3) / 4;       // float4 groups that hold the windows of 4 adjacent outputs
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x >= wl) return;
    const float* row = tmp + (size_t)blockIdx.z * tmp_stride + (size_t)y * Wp;
    const int a0 = S * x - NB - OFF;                    // a multiple of 4
    float u[4 * NV];
    if (a0 >= 0 && a0 + 4 * NV <= W) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(row + a0) + j);
            u[4 * j] = t.x; u[4 * j + 1] = t.y; u[4 * j + 2] = t.z; u[4 * j + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4 * NV; ++e) u[e] = row[reflect101(a0 + e, W)];
    }
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < T; ++j) acc = fmaf(wts.w[j], u[OFF + k * S + j], acc);
        o[k] = acc;
    }
    float* dst = img + (size_t)blockIdx.z * img_stride + (size_t)y * pitch + x;
    if (x + 4 <= wl) {
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x + k < wl) dst[k] = o[k];
    }
}

template <int LV>
__global__ void __launch_bounds__(128) pyr_hpass1_kernel(const float* __restrict__ tmp, size_t tmp_stride, int W, int Wp,
                                                        int wl, float* __restrict__ img, size_t img_stride, int pitch,
                                                        const __grid_constant__ HPassW wts) {
    pdl_entry();
    constexpr int S = HalfPyr::S(LV), T = HalfPyr::T(LV), NB = HalfPyr::NB(LV);
    constexpr int OFF = (4 - NB % 4) % 4;               // the window starts OFF floats into a 16-byte group
    constexpr int NV = (OFF + T + 3) / 4;
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= wl) return;
    const float* row = tmp + (size_t)blockIdx.z * tmp_stride + (size_t)y * Wp;
    const int a0 = S * x - NB - OFF;                    // a multiple of 4 (S is a multiple of 8)
    float acc = 0.f;
    if (a0 >= 0 && a0 + 4 * NV <= W) {
        const float4* q = reinterpret_cast<const float4*>(row + a0);
#pragma unroll
        for (int g = 0; g < NV; ++g) {
            const float4 t = __ldg(q + g);
            const float u[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (4 * g + e >= OFF && 4 * g + e - OFF < T) acc = fmaf(wts.w[4 * g + e - OFF], u[e], acc);
        }
    } else {
#pragma unroll 4
        for (int j = 0; j < T; ++j) acc = fmaf(wts.w[j], row[reflect101(a0 + OFF + j, W)], acc);
    }
    img[(size_t)blockIdx.z * img_stride + (size_t)y * pitch + x] = acc;
}

// level-0 image on its own (tests / taps only): 3x3 [1/4 1/2 1/4] blur of the u8 frame, REFLECT_101
__global__ void pyr0_kernel(const uint8_t* __restrict__ frame, int W, int H, float* __restrict__ img, int pitch) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= W) return;
    const float k[3] = {0.25f, 0.5f, 0.25f};
    float acc = 0.f;
    for (int dy = 0; dy < 3; ++dy)
        for (int dx = 0; dx < 3; ++dx)
            acc += k[dy] * k[dx] * (float)frame[(size_t)reflect101(y + dy - 1, H) * W + reflect101(x + dx - 1, W)];
    img[(size_t)y * pitch + x] = acc;
}

// ------------------------------------------------------------------------------------------------
// Polynomial expansion (FarnebackPolyExp).  64x32 output tile, halo 8 (poly_n <= 8), 256 threads.
//   staging         : float level image, or (U8) the raw u8 frame with the level-0 3x3 blur applied on
//                     the fly — all its products and sums are exact in float32, so the staged values are
//                     bit-identical to a separately blurred image
//   vertical pass   : thread = (column, 4 rows)  -> t0,t1,t2 in smem
//   horizontal pass : thread = (row, 4 columns)  -> float4 reads, float4 stores per plane
// ------------------------------------------------------------------------------------------------
constexpr int PE_TX = 64, PE_TY = 32, PE_H = 8, PE_RW = PE_TX + 2 * PE_H;  // 80

// horizontal [1/4 1/2 1/4] blur of four cells from the three aligned words around them (a holds the byte left of the
// first cell in its top byte, c the byte right of the last cell in its bottom byte).  Bytes -> floats with the
// mantissa trick (byte_to_float: permute + exact subtract, full-rate pipes) instead of I2F on the XU pipe.
__device__ __forceinline__ void blur3_words(uint32_t a, uint32_t b, uint32_t c, float (&hv)[4]) {
    const float v3 = byte_to_float(a, 0x7543u), v4 = byte_to_float(b, 0x7540u), v5 = byte_to_float(b, 0x7541u),
                v6 = byte_to_float(b, 0x7542u), v7 = byte_to_float(b, 0x7543u), v8 = byte_to_float(c, 0x7540u);
    hv[0] = 0.25f * v3 + 0.5f * v4 + 0.25f * v5;
    hv[1] = 0.25f * v4 + 0.5f * v5 + 0.25f * v6;
    hv[2] = 0.25f * v5 + 0.5f * v6 + 0.25f * v7;
    hv[3] = 0.25f * v6 + 0.5f * v7 + 0.25f * v8;
}

// The two separable passes of the expansion on a staged tile: raw[(PE_TY + 2 PE_H) x PE_RW] (row PE_H - n is the
// first staged row) -> t[3] (vertical sums) -> R.  Called by every polyexp kernel after its staging barrier.
template <int N_>
__device__ __forceinline__ void polyexp_passes(const float* __restrict__ raw, float (*t)[PE_TY * PE_RW], const PolyConst& pc,
                                               int n, int tid, int x0, int y0, int h, int pitch, float* __restrict__ R,
                                               size_t plane) {
    // vertical pass
    for (int task = tid; task < PE_RW * (PE_TY / 4); task += 256) {
        int c = task % PE_RW, g4 = task / PE_RW;
        float v[4 + 2 * PE_H];
#pragma unroll
        for (int j = 0; j < 4 + 2 * PE_H; ++j)
            v[j] = (j >= PE_H - n && j < 4 + PE_H + n) ? raw[(g4 * 4 + j) * PE_RW + c] : 0.f;
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            float a0 = v[PE_H + o] * pc.g[0], a1 = 0.f, a2 = 0.f;
#pragma unroll
            for (int k = 1; k <= kMaxPolyN; ++k) {
                if (k <= n) {
                    float up = v[PE_H + o - k], dn = v[PE_H + o + k];
                    float sum = up + dn;
                    a0 += pc.g[k] * sum;
                    a1 += pc.xg[k] * (dn - up);
                    a2 += pc.xxg[k] * sum;
                }
            }
            int r = g4 * 4 + o;
            t[0][r * PE_RW + c] = a0;
            t[1][r * PE_RW + c] = a1;
            t[2][r * PE_RW + c] = a2;
        }
    }
    __syncthreads();

    // horizontal pass
    for (int task = tid; task < PE_TY * (PE_TX / 4); task += 256) {
        int q = task % (PE_TX / 4), r = task / (PE_TX / 4);
        int y = y0 + r;
        if (y >= h) continue;
        float u0[4 + 2 * PE_H], u1[4 + 2 * PE_H], u2[4 + 2 * PE_H];
        const float4* p0 = reinterpret_cast<const float4*>(&t[0][r * PE_RW + 4 * q]);
        const float4* p1 = reinterpret_cast<const float4*>(&t[1][r * PE_RW + 4 * q]);
        const float4* p2 = reinterpret_cast<const float4*>(&t[2][r * PE_RW + 4 * q]);
#pragma unroll
        for (int j = 0; j < (4 + 2 * PE_H) / 4; ++j) {
            float4 a = p0[j], b = p1[j], c = p2[j];
            u0[4 * j] = a.x; u0[4 * j + 1] = a.y; u0[4 * j + 2] = a.z; u0[4 * j + 3] = a.w;
            u1[4 * j] = b.x; u1[4 * j + 1] = b.y; u1[4 * j + 2] = b.z; u1[4 * j + 3] = b.w;
            u2[4 * j] = c.x; u2[4 * j + 1] = c.y; u2[4 * j + 2] = c.z; u2[4 * j + 3] = c.w;
        }
        float o0[4], o1[4], o2[4], o3[4], o4[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            const int c = PE_H + o;
            float b1 = u0[c] * pc.g[0], b2 = 0.f, b3 = u1[c] * pc.g[0], b4 = 0.f, b5 = u2[c] * pc.g[0], b6 = 0.f;
#pragma unroll
            for (int k = 1; k <= kMaxPolyN; ++k) {
                if (k <= n) {
                    float tg = u0[c + k] + u0[c - k];
                    b1 += tg * pc.g[k];
                    b4 += tg * pc.xxg[k];
                    b2 += (u0[c + k] - u0[c - k]) * pc.xg[k];
                    b3 += (u1[c + k] + u1[c - k]) * pc.g[k];
                    b6 += (u1[c + k] - u1[c - k]) * pc.xg[k];
                    b5 += (u2[c + k] + u2[c - k]) * pc.g[k];
                }
            }
            o0[o] = b3 * pc.ig11;
            o1[o] = b2 * pc.ig11;
            o2[o] = b1 * pc.ig03 + b5 * pc.ig33;
            o3[o] = b1 * pc.ig03 + b4 * pc.ig33;
            o4[o] = b6 * pc.ig55;
        }
        float* dst = R + (size_t)y * pitch + x0 + 4 * q;
        *reinterpret_cast<float4*>(dst) = make_float4(o0[0], o0[1], o0[2], o0[3]);
        *reinterpret_cast<float4*>(dst + plane) = make_float4(o1[0], o1[1], o1[2], o1[3]);
        *reinterpret_cast<float4*>(dst + 2 * plane) = make_float4(o2[0], o2[1], o2[2], o2[3]);
        *reinterpret_cast<float4*>(dst + 3 * plane) = make_float4(o3[0], o3[1], o3[2], o3[3]);
        *reinterpret_cast<float4*>(dst + 4 * plane) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    }
}

// N_ > 0: poly_n known at compile time (5, 7 and 8 are instantiated: OpenCV's sample value, its other GPU value
// and the reference's) so the tap loops carry no predicates; N_ == 0: any poly_n <= 8 at run time.
template <bool U8, int N_>
__global__ void __launch_bounds__(256, 4) polyexp_kernel(const void* __restrict__ src_base, size_t src_stride, int w,
                                                     int h, int pitch, int u8_aligned, PolyConst pc,
                                                     float* __restrict__ R, size_t plane) {
    pdl_entry();
    __shared__ __align__(16) float raw[(PE_TY + 2 * PE_H) * PE_RW];
    __shared__ __align__(16) float t[3][PE_TY * PE_RW];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * PE_TX, y0 = blockIdx.y * PE_TY;
    const int n = N_ > 0 ? N_ : pc.n;

    // stage rows y0-n .. y0+TY+n-1 (replicate), columns x0-8 .. x0+TX+8-1 (replicate)
    const int rows = PE_TY + 2 * n;
    if (!U8) {
        const float* src = reinterpret_cast<const float*>(src_base) + (size_t)blockIdx.z * src_stride;
        for (int idx = tid; idx < rows * PE_RW; idx += 256) {
            int rr = idx / PE_RW, cc = idx - rr * PE_RW;
            int gy = clampi(y0 - n + rr, 0, h - 1);
            int gx = clampi(x0 - PE_H + cc, 0, w - 1);
            raw[(rr + PE_H - n) * PE_RW + cc] = src[(size_t)gy * pitch + gx];
        }
    } else {
        const uint8_t* src = reinterpret_cast<const uint8_t*>(src_base) + (size_t)blockIdx.z * src_stride;
        const bool fast = u8_aligned && (x0 - PE_H - 4 >= 0) && (x0 + PE_TX + PE_H + 4 <= w) && (y0 - n - 1 >= 0) &&
                          (y0 + PE_TY + n + 1 <= h);
        if (fast) {
            // 20 groups of 4 cells x 12 row segments.  Each thread first issues ALL its loads (three words per row,
            // rows r0-1 .. r1), then blurs: the global-load latency is paid once per thread, not once per row.
            constexpr int RPS_MAX = N_ > 0 ? (PE_TY + 2 * N_ + 11) / 12 : (PE_TY + 2 * kMaxPolyN + 11) / 12;
            const int g = tid % 20, seg = tid / 20;
            const int rps = (rows + 11) / 12;
            const int r0 = seg * rps, r1 = min(rows, r0 + rps);
            if (seg < 12 && r0 < r1) {
                const uint8_t* p = src + (size_t)(y0 - n + r0 - 1) * w + (x0 - PE_H + 4 * g - 4);
                uint32_t wa[RPS_MAX + 2], wb[RPS_MAX + 2], wc[RPS_MAX + 2];
#pragma unroll
                for (int i = 0; i < RPS_MAX + 2; ++i) {
                    if (i < r1 - r0 + 2) {
                        const uint32_t* q = reinterpret_cast<const uint32_t*>(p + (size_t)i * w);
                        wa[i] = __ldg(q); wb[i] = __ldg(q + 1); wc[i] = __ldg(q + 2);
                    } else {
                        wa[i] = wb[i] = wc[i] = 0u;
                    }
                }
                float hp[4], hc[4], hn[4];
                blur3_words(wa[0], wb[0], wc[0], hp);
                blur3_words(wa[1], wb[1], wc[1], hc);
#pragma unroll
                for (int i = 0; i < RPS_MAX; ++i) {
                    if (i < r1 - r0) {
                        blur3_words(wa[i + 2], wb[i + 2], wc[i + 2], hn);
                        float4 v;
                        v.x = 0.25f * hp[0] + 0.5f * hc[0] + 0.25f * hn[0];
                        v.y = 0.25f * hp[1] + 0.5f * hc[1] + 0.25f * hn[1];
                        v.z = 0.25f * hp[2] + 0.5f * hc[2] + 0.25f * hn[2];
                        v.w = 0.25f * hp[3] + 0.5f * hc[3] + 0.25f * hn[3];
                        *reinterpret_cast<float4*>(&raw[(r0 + i + PE_H - n) * PE_RW + 4 * g]) = v;
#pragma unroll
                        for (int k = 0; k < 4; ++k) { hp[k] = hc[k]; hc[k] = hn[k]; }
                    }
                }
            }
        } else {
            // border tiles: every staged row picks its own three source rows (replicated row for the expansion's
            // halo, REFLECT_101 neighbours for the 3x3 blur); groups of four cells whose three words lie inside the
            // row still use whole words, the few groups on the left / right image border go cell by cell
            const int g = tid % 20;
            const int gx0 = x0 - PE_H + 4 * g;
            const bool words = u8_aligned && gx0 - 4 >= 0 && gx0 + 8 <= w;
            for (int rr = tid / 20; rr < rows && tid < 240; rr += 12) {
                const int gy = clampi(y0 - n + rr, 0, h - 1);
                const int ym = reflect101(gy - 1, h), yp = reflect101(gy + 1, h);
                float4 v;
                if (words) {
                    const uint32_t* qa = reinterpret_cast<const uint32_t*>(src + (size_t)ym * w + (gx0 - 4));
                    const uint32_t* qb = reinterpret_cast<const uint32_t*>(src + (size_t)gy * w + (gx0 - 4));
                    const uint32_t* qc = reinterpret_cast<const uint32_t*>(src + (size_t)yp * w + (gx0 - 4));
                    float hp[4], hc[4], hn[4];
                    blur3_words(__ldg(qa), __ldg(qa + 1), __ldg(qa + 2), hp);
                    blur3_words(__ldg(qb), __ldg(qb + 1), __ldg(qb + 2), hc);
                    blur3_words(__ldg(qc), __ldg(qc + 1), __ldg(qc + 2), hn);
                    v.x = 0.25f * hp[0] + 0.5f * hc[0] + 0.25f * hn[0];
                    v.y = 0.25f * hp[1] + 0.5f * hc[1] + 0.25f * hn[1];
                    v.z = 0.25f * hp[2] + 0.5f * hc[2] + 0.25f * hn[2];
                    v.w = 0.25f * hp[3] + 0.5f * hc[3] + 0.25f * hn[3];
                } else {
                    const uint8_t *q0 = src + (size_t)ym * w, *q1 = src + (size_t)gy * w, *q2 = src + (size_t)yp * w;
                    float o[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int gx = clampi(gx0 + k, 0, w - 1);
                        const int xm = reflect101(gx - 1, w), xp = reflect101(gx + 1, w);
                        const float h0 = 0.25f * q0[xm] + 0.5f * q0[gx] + 0.25f * q0[xp];
                        const float h1 = 0.25f * q1[xm] + 0.5f * q1[gx] + 0.25f * q1[xp];
                        const float h2 = 0.25f * q2[xm] + 0.5f * q2[gx] + 0.25f * q2[xp];
                        o[k] = 0.25f * h0 + 0.5f * h1 + 0.25f * h2;
                    }
                    v = make_float4(o[0], o[1], o[2], o[3]);
                }
                *reinterpret_cast<float4*>(&raw[(rr + PE_H - n) * PE_RW + 4 * g]) = v;
            }
        }
    }
    __syncthreads();
    polyexp_passes<N_>(raw, t, pc, n, tid, x0, y0, h, pitch, R + (size_t)blockIdx.z * 5 * plane, plane);
}

// a global store whose address space survives the register pinning of the base pointer below (a plain store through
// a pointer that went through an asm operand would be emitted as a generic ST)
__device__ __forceinline__ void st_global_f32(float* p, float v) {
    asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v));
}

// ------------------------------------------------------------------------------------------------
// FarnebackUpdateMatrices for one pixel.  R0/R1 point at plane 0 of the two frames' expansions.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float border_factor(int d) { return d < 2 ? 0.14f : 0.4472f; }

struct R0Px { float y, x, yy, xx, xy; };     // the five expansion coefficients of one pixel of the first frame

__device__ __forceinline__ R0Px load_r0_px(const float* __restrict__ R0, size_t o, size_t plane) {
    R0Px r;
    r.y = __ldg(R0 + o); r.x = __ldg(R0 + plane + o); r.yy = __ldg(R0 + 2 * plane + o);
    r.xx = __ldg(R0 + 3 * plane + o); r.xy = __ldg(R0 + 4 * plane + o);
    return r;
}

__device__ __forceinline__ void update_matrices_px(int x, int y, int w, int h, int pitch, size_t plane, float dx,
                                                   float dy, const R0Px& r0,
                                                   const float* __restrict__ R1, float* __restrict__ Mout) {
    const size_t o = (size_t)y * pitch + x;
    const float r0y = r0.y, r0x = r0.x, r0yy = r0.yy, r0xx = r0.xx, r0xy = r0.xy;
    float fx = (float)x + dx, fy = (float)y + dy;
    const float flx = floorf(fx), fly = floorf(fy);
    // keep the int conversion safe for wild displacements
    const int x1 = (int)fminf(fmaxf(flx, -2.f), 1.0e6f), y1 = (int)fminf(fmaxf(fly, -2.f), 1.0e6f);
    fx -= flx;
    fy -= fly;
    float r2, r3, r4, r5, r6;
    if ((unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1)) {
        const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
        const float* p = R1 + (size_t)y1 * pitch + x1;
        r2 = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(p + pitch) + a11 * __ldg(p + pitch + 1);
        p += plane;
        r3 = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(p + pitch) + a11 * __ldg(p + pitch + 1);
        p += plane;
        r4 = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(p + pitch) + a11 * __ldg(p + pitch + 1);
        p += plane;
        r5 = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(p + pitch) + a11 * __ldg(p + pitch + 1);
        p += plane;
        r6 = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(p + pitch) + a11 * __ldg(p + pitch + 1);
        r4 = (r0yy + r4) * 0.5f;
        r5 = (r0xx + r5) * 0.5f;
        r6 = (r0xy + r6) * 0.25f;
    } else {
        r2 = r3 = 0.f;
        r4 = r0yy;
        r5 = r0xx;
        r6 = r0xy * 0.5f;
    }
    r2 = (r0y - r2) * 0.5f;
    r3 = (r0x - r3) * 0.5f;
    r2 += r4 * dy + r6 * dx;
    r3 += r6 * dy + r5 * dx;
    if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
        const float sc = (x < 5 ? border_factor(x) : 1.f) * (x >= w - 5 ? border_factor(w - x - 1) : 1.f) *
                         (y < 5 ? border_factor(y) : 1.f) * (y >= h - 5 ? border_factor(h - y - 1) : 1.f);
        r2 *= sc; r3 *= sc; r4 *= sc; r5 *= sc; r6 *= sc;
    }
    Mout[o] = r4 * r4 + r6 * r6;
    Mout[plane + o] = (r4 + r5) * r6;
    Mout[2 * plane + o] = r5 * r5 + r6 * r6;
    Mout[3 * plane + o] = r4 * r2 + r6 * r3;
    Mout[4 * plane + o] = r6 * r2 + r5 * r3;
}

// Level entry: flow_l = resize(flow_{l+1}) * (1/pyr_scale) (zeros on the coarsest level), then
// UpdateMatrices.  The upsampled flow itself is never stored: BlurBox rebuilds the flow from M alone.
// cv::resize(INTER_LINEAR) source index / weight of destination index d (api.cu: resize_tables), evaluated with the
// same double operations, one rounding each, so the values equal the host-built tables bit for bit
__device__ __forceinline__ void resize_coord(int d, double scale, int src, int& i0, float& a) {
    const float f = (float)__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5);
    int s = (int)floorf(f);
    a = f - (float)s;
    if (s < 0) { s = 0; a = 0.f; }
    if (s >= src - 1) { s = src - 1; a = 0.f; }
    i0 = s;
}

// COORD selects how the resize coordinates are obtained: 0 = recomputed with resize_coord's double operations,
// 1 = read from the host-built tables, 2 = recomputed in float32, valid (and bit-identical) when both scales are
// powers of two, e.g. 1920 -> 960: (d + 0.5) * 2^-k - 0.5 is then exact in float32 as well
enum { MI_COORD_F64 = 0, MI_COORD_TABLES = 1, MI_COORD_POW2 = 2 };

__device__ __forceinline__ void resize_coord_pow2(int d, float scale, int src, int& i0, float& a) {
    const float f = __fsub_rn(__fmul_rn(__fadd_rn((float)d, 0.5f), scale), 0.5f);
    int s = (int)floorf(f);
    a = f - (float)s;
    if (s < 0) { s = 0; a = 0.f; }
    if (s >= src - 1) { s = src - 1; a = 0.f; }
    i0 = s;
}

constexpr int MI_TX = 64, MI_TY = 4;   // matrices_init_kernel block: 64 x 4 pixels

template <int COORD>
__global__ void __launch_bounds__(256, 8) matrices_init_kernel(const float* __restrict__ R, size_t plane, int w, int h,
                                                           int pitch, size_t R_pair_stride,
                                                           const float2* __restrict__ cflow, int cw, int ch,
                                                           int cpitch, size_t cflow_stride,
                                                           const int* __restrict__ fxi0,
                                                           const float* __restrict__ fxa,
                                                           const int* __restrict__ fyi0,
                                                           const float* __restrict__ fya, float up_scale,
                                                           float* __restrict__ M, double xscale, double yscale, int r0_first) {
    pdl_entry();
    // 3-D grid (pairs, tiles_x, tiles_y): blocks are scheduled x-fastest, so the pair index is fastest (same L2 sharing
    // of R between consecutive pairs as in iter_box_tma_kernel) and no thread pays for an integer division: with one
    // pixel per thread the two divisions of a 1-D grid were 55 of the kernel's 400 instructions
    const int p = blockIdx.x;
    const int x = blockIdx.y * MI_TX + (threadIdx.x & (MI_TX - 1));
    const int y = blockIdx.z * MI_TY + threadIdx.x / MI_TX;
    if (x >= w || y >= h) return;
    // R0 does not depend on the flow: its five loads go out first and travel with the coarse-flow loads, so that the
    // second memory round trip of the thread is the R1 gather alone.  The host always passes r0_first = 1.  The order
    // stays a run-time branch because the compile-time form (R0 loaded first, no second load site) is slower: 2.15 vs
    // 2.05 ms per C2 step (B200, 1000 W).  With the order fixed, ptxas keeps the 64-bit pixel offset live from the R0
    // loads to the M stores and issues the R1 gather in smaller groups.
    const float* R0 = R + (size_t)p * R_pair_stride;
    R0Px r0;
    if (r0_first) r0 = load_r0_px(R0, (size_t)y * pitch + x, plane);
    float dx = 0.f, dy = 0.f;
    if (cflow) {
        const float2* cf = cflow + (size_t)p * cflow_stride;
        int xa0, ya0;
        float ax, ay;
        if (COORD == MI_COORD_TABLES) {
            xa0 = fxi0[x]; ya0 = fyi0[y]; ax = fxa[x]; ay = fya[y];
        } else if (COORD == MI_COORD_POW2) {
            resize_coord_pow2(x, (float)xscale, cw, xa0, ax);
            resize_coord_pow2(y, (float)yscale, ch, ya0, ay);
        } else {
            // one dependent memory round trip less than reading the tables
            resize_coord(x, xscale, cw, xa0, ax);
            resize_coord(y, yscale, ch, ya0, ay);
        }
        const int xa1 = min(xa0 + 1, cw - 1), ya1 = min(ya0 + 1, ch - 1);
        const float2 f00 = cf[(size_t)ya0 * cpitch + xa0], f01 = cf[(size_t)ya0 * cpitch + xa1];
        const float2 f10 = cf[(size_t)ya1 * cpitch + xa0], f11 = cf[(size_t)ya1 * cpitch + xa1];
        const float tx0 = f00.x * (1.f - ax) + f01.x * ax, tx1 = f10.x * (1.f - ax) + f11.x * ax;
        const float ty0 = f00.y * (1.f - ax) + f01.y * ax, ty1 = f10.y * (1.f - ax) + f11.y * ax;
        dx = (tx0 * (1.f - ay) + tx1 * ay) * up_scale;
        dy = (ty0 * (1.f - ay) + ty1 * ay) * up_scale;
    }
    if (!r0_first) r0 = load_r0_px(R0, (size_t)y * pitch + x, plane);
    // One pixel per thread at 32 registers (full occupancy) is the fastest form measured: the 32-bit-offset
    // UpdateMatrices of the fused iteration (> 32 registers: 0.87 vs 0.675 ms per 16-pair step) and variants with
    // 8 pixels per thread that halve the instruction count (2.45-2.67 vs 2.22 ms per 64-pair step), and a tiled
    // variant with the R1 footprint staged by TMA like the fused iteration's (2.57 ms), all lose more to occupancy
    // than they save: the kernel is bound by the latency of its dependent memory round trips.  Round 2 repeated the
    // experiment at 32 registers (unsigned 32-bit element offsets from pinned base pointers, one IMAD.WIDE.U32 per
    // address, 352 instead of 384 SASS instructions, no spills): 2.20 vs 2.04 ms per 64-pair step — slower again.
    update_matrices_px(x, y, w, h, pitch, plane, dx, dy, r0, R0 + 5 * plane, M + (size_t)p * 5 * plane);
}

// ------------------------------------------------------------------------------------------------
// Fused iteration: flow = solve(blur(M));  M' = UpdateMatrices(R0, R1, flow).
// 64x32 tile, 256 threads.  The five planes of M are blurred one after the other through a small
// smem staging area (raw tile + vertical sums); the blurred sums land in S[5][32][64]; the final
// phase is per pixel with x fastest so R0 loads, the R1 gather and the M' stores are coalesced.
// ------------------------------------------------------------------------------------------------
constexpr int IT_TX = 64, IT_TY = 32;
// Consecutive pairs share an R plane (R1 of pair p is R0 of pair p+1): iter_box_tma_kernel interleaves the pairs of a
// tile in groups of 4 in its CTA order so that the second reader hits L2 (4502 vs 4441 pairs/s ungrouped, 4338 with the
// whole 64-pair batch interleaved: too many concurrent HBM regions).
constexpr int IT_PAIR_GROUP = 4;

struct IterArgs {
    const float* Min;
    float* Mout;
    const float* R;
    float2* flow;           // nullable
    int flow_pitch;         // float2 units
    size_t flow_stride;     // float2 units per pair
    int w, h, pitch;
    size_t plane;
    int m;                  // winsize / 2
    int hx;                 // column halo, m rounded up to a multiple of 4
    float scale;            // 1 / winsize^2 (box) or 1 (Gaussian: kernel already normalised)
    int pair_stride;
    const float* gk;        // Gaussian half kernel [m+1] (device) or nullptr
    int n_pairs, tiles_x;   // TMA kernel: 1-D grid (see iter_box_tma_kernel)
};

template <int M_>
__device__ __forceinline__ void hsum_box(const float (&u)[20], float (&o)[4]) {
    // window for output j covers u[8 - M_ + j .. 8 + M_ + j]
    float s = 0.f;
#pragma unroll
    for (int j = 8 - M_; j <= 8 + M_; ++j) s += u[j];
    o[0] = s;
#pragma unroll
    for (int j = 1; j < 4; ++j) {
        s += u[8 + M_ + j] - u[8 - M_ + j - 1];
        o[j] = s;
    }
}

template <int M_>
__device__ __forceinline__ void hsum_gauss(const float (&u)[20], const float* __restrict__ gk, float (&o)[4]) {
    float k[M_ + 1];
#pragma unroll
    for (int i = 0; i <= M_; ++i) k[i] = gk[i];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        // explicit multiply / fused multiply-add: every kernel that evaluates this filter rounds identically
        float s = __fmul_rn(u[8 + j], k[0]);
#pragma unroll
        for (int i = 1; i <= M_; ++i) s = __fmaf_rn(u[8 + j - i] + u[8 + j + i], k[i], s);
        o[j] = s;
    }
}

template <int M_>
__device__ __forceinline__ void hsum_gauss_reg(const float (&u)[20], const float (&k)[M_ + 1], float (&o)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float s = __fmul_rn(u[8 + j], k[0]);
#pragma unroll
        for (int i = 1; i <= M_; ++i) s = __fmaf_rn(u[8 + j - i] + u[8 + j + i], k[i], s);
        o[j] = s;
    }
}

template <bool GAUSS, bool LAST>
__global__ void __launch_bounds__(256, 3) iter_kernel(IterArgs a) {
    pdl_entry();
    extern __shared__ __align__(16) float smem[];
    const int m = a.m, hx = a.hx;
    const int RW = IT_TX + 2 * hx;          // staged columns
    const int RH = IT_TY + 2 * m;           // staged rows
    float* raw = smem;                      // [RH][RW]
    float* vs = raw + RH * RW;              // [IT_TY][RW]
    float* S = vs + IT_TY * RW;             // [5][IT_TY][IT_TX]
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * IT_TX, y0 = blockIdx.y * IT_TY;
    const int p = blockIdx.z;
    const int w = a.w, h = a.h, pitch = a.pitch;
    const size_t plane = a.plane;
    const float* Min = a.Min + (size_t)p * 5 * plane;
    const bool interior = (x0 - hx >= 0) && (x0 + IT_TX + hx <= w) && (y0 - m >= 0) && (y0 + IT_TY + m <= h);

    for (int c = 0; c < 5; ++c) {
        const float* src = Min + c * plane;
        // ---- stage the tile + halo (replicate borders) ----
        if (interior) {
            const int n4 = RW >> 2;
            const float* base = src + (size_t)(y0 - m) * pitch + (x0 - hx);
            for (int idx = tid; idx < RH * n4; idx += 256) {
                int rr = idx / n4, q = idx - rr * n4;
                float4 v = __ldg(reinterpret_cast<const float4*>(base + (size_t)rr * pitch) + q);
                *reinterpret_cast<float4*>(raw + rr * RW + 4 * q) = v;
            }
        } else {
            for (int idx = tid; idx < RH * RW; idx += 256) {
                int rr = idx / RW, cc = idx - rr * RW;
                int gy = clampi(y0 - m + rr, 0, h - 1);
                int gx = clampi(x0 - hx + cc, 0, w - 1);
                raw[idx] = __ldg(src + (size_t)gy * pitch + gx);
            }
        }
        __syncthreads();
        // ---- vertical pass over the columns that are needed: [hx-m, hx+TX+m) ----
        const int ncols = IT_TX + 2 * m;
        if (!GAUSS) {
            // running sums, 4 segments of 8 rows per column
            for (int task = tid; task < ncols * 4; task += 256) {
                int cc = task % ncols + (hx - m), seg = task / ncols;
                const float* col = raw + (seg * 8) * RW + cc;
                float s = 0.f;
                for (int j = 0; j <= 2 * m; ++j) s += col[j * RW];
                float* dst = vs + (seg * 8) * RW + cc;
                dst[0] = s;
#pragma unroll
                for (int o = 1; o < 8; ++o) {
                    s += col[(o + 2 * m) * RW] - col[(o - 1) * RW];
                    dst[o * RW] = s;
                }
            }
        } else {
            for (int task = tid; task < ncols * IT_TY; task += 256) {
                int cc = task % ncols + (hx - m), r = task / ncols;
                const float* col = raw + r * RW + cc;
                float s = __fmul_rn(col[m * RW], __ldg(a.gk));
                for (int i = 1; i <= m; ++i) s = __fmaf_rn(col[(m - i) * RW] + col[(m + i) * RW], __ldg(a.gk + i), s);
                vs[r * RW + cc] = s;
            }
        }
        __syncthreads();
        // ---- horizontal pass: thread = (row, 4 columns) ----
        float* Sc = S + c * (IT_TY * IT_TX);
        if (hx == 8 && m >= 5) {
            for (int task = tid; task < IT_TY * (IT_TX / 4); task += 256) {
                int q = task & 15, r = task >> 4;
                const float4* pv = reinterpret_cast<const float4*>(vs + r * RW + 4 * q);
                float u[20];
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    float4 v = pv[j];
                    u[4 * j] = v.x; u[4 * j + 1] = v.y; u[4 * j + 2] = v.z; u[4 * j + 3] = v.w;
                }
                float o[4];
                if (!GAUSS) {
                    switch (m) {
                        case 5: hsum_box<5>(u, o); break;
                        case 6: hsum_box<6>(u, o); break;
                        case 7: hsum_box<7>(u, o); break;
                        default: hsum_box<8>(u, o); break;
                    }
                } else {
                    switch (m) {
                        case 5: hsum_gauss<5>(u, a.gk, o); break;
                        case 6: hsum_gauss<6>(u, a.gk, o); break;
                        case 7: hsum_gauss<7>(u, a.gk, o); break;
                        default: hsum_gauss<8>(u, a.gk, o); break;
                    }
                }
                *reinterpret_cast<float4*>(Sc + r * IT_TX + 4 * q) = make_float4(o[0], o[1], o[2], o[3]);
            }
        } else {
            // generic window: one pixel per thread step, conflict-free scalar reads
            for (int idx = tid; idx < IT_TY * IT_TX; idx += 256) {
                int cx = idx & 63, r = idx >> 6;
                const float* row = vs + r * RW + hx + cx;
                float s;
                if (!GAUSS) {
                    s = 0.f;
                    for (int j = -m; j <= m; ++j) s += row[j];
                } else {
                    s = __fmul_rn(row[0], __ldg(a.gk));
                    for (int i = 1; i <= m; ++i) s = __fmaf_rn(row[-i] + row[i], __ldg(a.gk + i), s);
                }
                Sc[idx] = s;
            }
        }
        // the next channel's staging writes `raw` (last read before the previous barrier) and its
        // vertical pass writes `vs` only after the barrier that follows staging -> no extra barrier
    }
    __syncthreads();

    // ---- per-pixel solve + matrix update (x fastest) ----
    const float* R0 = a.R + (size_t)(p * a.pair_stride) * 5 * plane;
    const float* R1 = R0 + 5 * plane;
    float* Mout = LAST ? nullptr : a.Mout + (size_t)p * 5 * plane;
#pragma unroll 2
    for (int j = 0; j < (IT_TX * IT_TY) / 256; ++j) {
        const int idx = j * 256 + tid;
        const int cx = idx & 63, r = idx >> 6;
        const int x = x0 + cx, y = y0 + r;
        if (x >= w || y >= h) continue;
        const float g11 = S[idx] * a.scale, g12 = S[IT_TX * IT_TY + idx] * a.scale,
                    g22 = S[2 * IT_TX * IT_TY + idx] * a.scale, h1 = S[3 * IT_TX * IT_TY + idx] * a.scale,
                    h2 = S[4 * IT_TX * IT_TY + idx] * a.scale;
        const float idet = 1.f / (g11 * g22 - g12 * g12 + 1e-3f);
        const float fx = (g11 * h2 - g12 * h1) * idet;
        const float fy = (g22 * h1 - g12 * h2) * idet;
        if (a.flow) a.flow[(size_t)p * a.flow_stride + (size_t)y * a.flow_pitch + x] = make_float2(fx, fy);
        if (!LAST) update_matrices_px(x, y, w, h, pitch, plane, fx, fy, load_r0_px(R0, (size_t)y * pitch + x, plane), R1, Mout);
    }
}

// ------------------------------------------------------------------------------------------------
// Fused iteration, TMA-staged (box window, 5 <= m <= 8): the production path.
//
// One cp.async.bulk.tensor (TMA) brings the 5 x (32+2m) x 80 float box of M — all five planes of the
// tile plus halo — into shared memory; everything after that happens IN PLACE in that box:
//   vertical   thread = (plane, column): running 2m+1 sum marching down the column, window in
//              registers, the sum for row y overwrites row y after its input has been consumed
//   horizontal thread = 4 adjacent pixels of one row: the five planes' sums from 5 float4 reads each and
//              the 2x2 solve, in registers
//   pixel      (not the last iteration) the flow vectors pass through shared memory to an x-fastest mapping;
//              then a SECOND TMA load puts the five R1 planes around the tile (displaced by the tile centre's
//              flow) into the same box, and UpdateMatrices gathers from shared memory (global fallback for
//              footprints outside the box), with coalesced R0 loads and M' stores
// Out-of-image box cells arrive as zeros (TMA fill) and are overwritten with the replicated edge
// values for border tiles only.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}

// L2 prefetch of a tensor box (no shared memory, no completion tracking)
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
                 ::"l"(map), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Polynomial expansion with the tile staged by TMA (tuning.polyexp_tma, default): ONE cp.async.bulk.tensor brings the
// tile + halo into shared memory — the u8 frame box {96 bytes, 34 + 2n rows} for level 0, the float image box
// {80, 32 + 2n} for the coarser levels — instead of every thread issuing (and waiting for) its own global loads.
// Level 0 then applies the 3x3 [1/4 1/2 1/4] blur from shared-memory words; out-of-image cells arrive as zeros and are
// fixed up for border tiles only: the one-pixel REFLECT_101 ring the blur reads, then (on the blurred floats) the
// replicated rows / columns the expansion reads.  Arithmetic and its order are those of polyexp_kernel: bit-identical R.
// ------------------------------------------------------------------------------------------------
constexpr int PE_BW = 96;   // bytes per staged u8 row: x0 - 16 .. x0 + 79 (16-byte aligned box origin)

template <bool U8, int N_>
__global__ void __launch_bounds__(256, 4) polyexp_tma_kernel(const __grid_constant__ CUtensorMap tmap, int w, int h,
                                                         int pitch, PolyConst pc, float* __restrict__ R, size_t plane) {
    pdl_entry();
    __shared__ __align__(128) float raw[(PE_TY + 2 * PE_H) * PE_RW];
    __shared__ __align__(128) float t[3][PE_TY * PE_RW];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * PE_TX, y0 = blockIdx.y * PE_TY;
    const int n = N_ > 0 ? N_ : pc.n;
    const int rows = PE_TY + 2 * n;
    // level 0: the byte box is parked in the (not yet used) vertical-sum area: (rows + 2) x 96 bytes <= 50 x 96
    uint8_t* bytes = reinterpret_cast<uint8_t*>(&t[0][0]);
    float* raw0 = raw;                                      // first staged row (TMA destination: 128-byte aligned)
    if (tid == 0) {
        mbar_init(&bar, 1);
        if (U8) {
            mbar_expect_tx(&bar, (uint32_t)((rows + 2) * PE_BW));
            tma_load_3d(bytes, &tmap, x0 - 16, y0 - n - 1, blockIdx.z, &bar);
        } else {
            mbar_expect_tx(&bar, (uint32_t)(rows * PE_RW * sizeof(float)));
            tma_load_3d(raw0, &tmap, x0 - PE_H, y0 - n, blockIdx.z, &bar);
        }
    }
    const bool interior = (x0 - PE_H - 1 >= 0) && (x0 + PE_TX + PE_H + 1 <= w) && (y0 - n - 1 >= 0) &&
                          (y0 + PE_TY + n + 1 <= h);
    __syncthreads();
    mbar_wait(&bar, 0);
    if (U8) {
        if (!interior) {
            // REFLECT_101 ring of the source: column -1 <- 1, column w <- w - 2, then row -1 <- 1, row h <- h - 2
            // (cells further out are never read by the blur of an in-image pixel)
            for (int rr = tid; rr < rows + 2; rr += 256) {
                uint8_t* row = bytes + rr * PE_BW;
                const int bl = -1 - (x0 - 16), br = w - (x0 - 16);          // box columns of x = -1 and x = w
                if (bl >= 0 && bl + 2 < PE_BW) row[bl] = row[bl + 2];
                if (br >= 2 && br < PE_BW) row[br] = row[br - 2];
            }
            __syncthreads();
            for (int cc = tid; cc < PE_BW; cc += 256) {
                const int bt = -1 - (y0 - n - 1), bb = h - (y0 - n - 1);    // box rows of y = -1 and y = h
                if (bt >= 0 && bt + 2 < rows + 2) bytes[bt * PE_BW + cc] = bytes[(bt + 2) * PE_BW + cc];
                if (bb >= 2 && bb < rows + 2) bytes[bb * PE_BW + cc] = bytes[(bb - 2) * PE_BW + cc];
            }
            __syncthreads();
        }
        // blur: 20 groups of 4 cells x 12 row segments; staged row rr, cell cc = box row rr + 1, box byte cc + 8
        const int g = tid % 20, seg = tid / 20;
        const int rps = (rows + 11) / 12;
        const int r0 = seg * rps, r1 = min(rows, r0 + rps);
        if (seg < 12 && r0 < r1) {
            const uint32_t* wp = reinterpret_cast<const uint32_t*>(bytes + r0 * PE_BW + 4 * g + 4);   // word left of the cells
            float hp[4], hc[4], hn[4];
            blur3_words(wp[0], wp[1], wp[2], hp);
            blur3_words(wp[PE_BW / 4], wp[PE_BW / 4 + 1], wp[PE_BW / 4 + 2], hc);
            for (int i = 0; i < r1 - r0; ++i) {
                const uint32_t* q = wp + (i + 2) * (PE_BW / 4);
                blur3_words(q[0], q[1], q[2], hn);
                float4 v;
                v.x = 0.25f * hp[0] + 0.5f * hc[0] + 0.25f * hn[0];
                v.y = 0.25f * hp[1] + 0.5f * hc[1] + 0.25f * hn[1];
                v.z = 0.25f * hp[2] + 0.5f * hc[2] + 0.25f * hn[2];
                v.w = 0.25f * hp[3] + 0.5f * hc[3] + 0.25f * hn[3];
                *reinterpret_cast<float4*>(&raw0[(r0 + i) * PE_RW + 4 * g]) = v;
#pragma unroll
                for (int k = 0; k < 4; ++k) { hp[k] = hc[k]; hc[k] = hn[k]; }
            }
        }
        __syncthreads();          // the byte box (in t) is dead from here on; raw is complete for in-image cells
    }
    if (!interior) {
        // the expansion reads replicated rows / columns: out-of-image cells take the clamped cell's value (columns
        // beside the image on the in-image rows first, then whole rows above / below it)
        const int xlo = max(0, PE_H - x0), xhi = min(PE_RW, w - x0 + PE_H);      // in-image columns [xlo, xhi)
        const int ylo = max(0, n - y0), yhi = min(rows, h - y0 + n);             // in-image rows [ylo, yhi)
        const int ncol = xlo + (PE_RW - xhi);
        if (ncol > 0) {
            for (int idx = tid; idx < (yhi - ylo) * ncol; idx += 256) {
                const int rr = ylo + idx / ncol, k = idx % ncol;
                float* row = raw0 + rr * PE_RW;
                row[k < xlo ? k : xhi + (k - xlo)] = row[k < xlo ? xlo : xhi - 1];
            }
            __syncthreads();
        }
        const int nrow_out = ylo + (rows - yhi);
        if (nrow_out > 0) {
            for (int idx = tid; idx < nrow_out * (PE_RW / 4); idx += 256) {
                const int k = idx / (PE_RW / 4), q = idx - k * (PE_RW / 4);
                const int rr = k < ylo ? k : yhi + (k - ylo);
                reinterpret_cast<float4*>(raw0 + rr * PE_RW)[q] =
                    reinterpret_cast<const float4*>(raw0 + (k < ylo ? ylo : yhi - 1) * PE_RW)[q];
            }
            __syncthreads();
        }
    }
    // the passes address the tile with its first staged row at row PE_H - n
    polyexp_passes<N_>(raw0 - (PE_H - n) * PE_RW, t, pc, n, tid, x0, y0, h, pitch, R + (size_t)blockIdx.z * 5 * plane, plane);
}

// UpdateMatrices with the R1 footprint read from a shared-memory box [5][RH][RW] whose cell (0, 0) is image pixel
// (bx, by); footprints that leave the box fall back to global loads.  `edge` is tile-uniform (tile within 5 px of a
// border).  Same operations, same order as update_matrices_px (the generic iter_kernel's): identical results.

__device__ __forceinline__ R0Px load_r0(const float* __restrict__ R0, unsigned o, unsigned plane) {
    R0Px r;
    r.y = __ldg(R0 + o); r.x = __ldg(R0 + (o + plane)); r.yy = __ldg(R0 + (o + 2 * plane));
    r.xx = __ldg(R0 + (o + 3 * plane)); r.xy = __ldg(R0 + (o + 4 * plane));
    return r;
}

template <int RW, int RH>
__device__ __forceinline__ void update_matrices_box(int x, int y, int w, int h, int pitch, unsigned plane, bool edge, float dx,
                                                    float dy, const R0Px& r0, const float* __restrict__ R1,
                                                    float* __restrict__ Mout, const float* box, int bx, int by) {
    constexpr int CH = RH * RW;
    const unsigned o = (unsigned)(y * pitch + x);       // unsigned element offsets: one IMAD.WIDE.U32 per address
    const float r0y = r0.y, r0x = r0.x, r0yy = r0.yy, r0xx = r0.xx, r0xy = r0.xy;
    float fx = (float)x + dx, fy = (float)y + dy;
    const float flx = floorf(fx), fly = floorf(fy);
    const int x1 = (int)fminf(fmaxf(flx, -2.f), 1.0e6f), y1 = (int)fminf(fmaxf(fly, -2.f), 1.0e6f);
    fx -= flx;
    fy -= fly;
    float r2, r3, r4, r5, r6;
    if ((unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1)) {
        const float gx = 1.f - fx, gy = 1.f - fy;
        const float a00 = gx * gy, a01 = fx * gy, a10 = gx * fy, a11 = fx * fy;
        const int lx = x1 - bx, ly = y1 - by;
        if ((unsigned)lx < (unsigned)(RW - 1) && (unsigned)ly < (unsigned)(RH - 1)) {
            const float* q = box + ly * RW + lx;
            r2 = a00 * q[0] + a01 * q[1] + a10 * q[RW] + a11 * q[RW + 1];
            r3 = a00 * q[CH] + a01 * q[CH + 1] + a10 * q[CH + RW] + a11 * q[CH + RW + 1];
            r4 = a00 * q[2 * CH] + a01 * q[2 * CH + 1] + a10 * q[2 * CH + RW] + a11 * q[2 * CH + RW + 1];
            r5 = a00 * q[3 * CH] + a01 * q[3 * CH + 1] + a10 * q[3 * CH + RW] + a11 * q[3 * CH + RW + 1];
            r6 = a00 * q[4 * CH] + a01 * q[4 * CH + 1] + a10 * q[4 * CH + RW] + a11 * q[4 * CH + RW + 1];
        } else {
            const unsigned q0 = (unsigned)(y1 * pitch + x1), q1 = q0 + (unsigned)pitch;
            r2 = a00 * __ldg(R1 + q0) + a01 * __ldg(R1 + q0 + 1) + a10 * __ldg(R1 + q1) + a11 * __ldg(R1 + q1 + 1);
            r3 = a00 * __ldg(R1 + (q0 + plane)) + a01 * __ldg(R1 + (q0 + plane) + 1) +
                 a10 * __ldg(R1 + (q1 + plane)) + a11 * __ldg(R1 + (q1 + plane) + 1);
            r4 = a00 * __ldg(R1 + (q0 + 2 * plane)) + a01 * __ldg(R1 + (q0 + 2 * plane) + 1) +
                 a10 * __ldg(R1 + (q1 + 2 * plane)) + a11 * __ldg(R1 + (q1 + 2 * plane) + 1);
            r5 = a00 * __ldg(R1 + (q0 + 3 * plane)) + a01 * __ldg(R1 + (q0 + 3 * plane) + 1) +
                 a10 * __ldg(R1 + (q1 + 3 * plane)) + a11 * __ldg(R1 + (q1 + 3 * plane) + 1);
            r6 = a00 * __ldg(R1 + (q0 + 4 * plane)) + a01 * __ldg(R1 + (q0 + 4 * plane) + 1) +
                 a10 * __ldg(R1 + (q1 + 4 * plane)) + a11 * __ldg(R1 + (q1 + 4 * plane) + 1);
        }
        r4 = (r0yy + r4) * 0.5f;
        r5 = (r0xx + r5) * 0.5f;
        r6 = (r0xy + r6) * 0.25f;
    } else {
        r2 = r3 = 0.f;
        r4 = r0yy;
        r5 = r0xx;
        r6 = r0xy * 0.5f;
    }
    r2 = (r0y - r2) * 0.5f;
    r3 = (r0x - r3) * 0.5f;
    r2 += r4 * dy + r6 * dx;
    r3 += r6 * dy + r5 * dx;
    if (edge && ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10))) {
        const float sc = (x < 5 ? border_factor(x) : 1.f) * (x >= w - 5 ? border_factor(w - x - 1) : 1.f) *
                         (y < 5 ? border_factor(y) : 1.f) * (y >= h - 5 ? border_factor(h - y - 1) : 1.f);
        r2 *= sc; r3 *= sc; r4 *= sc; r5 *= sc; r6 *= sc;
    }
    st_global_f32(Mout + o, r4 * r4 + r6 * r6);
    st_global_f32(Mout + (o + plane), (r4 + r5) * r6);
    st_global_f32(Mout + (o + 2 * plane), r5 * r5 + r6 * r6);
    st_global_f32(Mout + (o + 3 * plane), r4 * r2 + r6 * r3);
    st_global_f32(Mout + (o + 4 * plane), r6 * r2 + r5 * r3);
}

// Not-last iterations: the horizontal sums and the solve are done in registers as in the last iteration and the flow
// vectors, not the five sums, go through shared memory to reach the x-fastest pixel mapping of the update phase (640 ->
// 256 wavefronts per tile for that hand-over, one more barrier: 4.27 vs 4.39 ms per 64-pair step against writing the
// sums back to the box; same hsum_box, same solve expressions: identical results).  (A variant that parked the flow
// vectors in the dead raw rows below the vertical sums to save that barrier measured 0.5 % slower and was removed.)
// R1 is staged in shared memory by the second TMA load: 4.36 vs 4.56 ms per 64-pair step against gathering it from
// global memory.
// TY: tile height, 32 by default; 16 for launches whose 32-row tiling would leave SMs idle (single pairs, the coarse
// levels): twice the CTAs, half the serial work per CTA.  The vertical sums are re-seeded at absolute rows that are
// multiples of 8 in both tilings and the horizontal groups start at multiples of 4: the results are bit-identical.
// GAUSS: OPTFLOW_FARNEBACK_GAUSSIAN windows (FarnebackUpdateFlow_GaussianBlur): the vertical pass is the 2m+1-tap
// filter on the same register window (in place, like the running sums), the horizontal one hsum_gauss; both with the
// generic kernel's expressions, so the two kernels stay bit-identical.
template <int M_, bool LAST, int TY, bool GAUSS>
__global__ void __launch_bounds__(256, 3) iter_box_tma_kernel(const __grid_constant__ CUtensorMap tmap,
                                                              const __grid_constant__ CUtensorMap tmapR,
                                                              const __grid_constant__ CUtensorMap tmapRbox, IterArgs a) {
    pdl_entry();
    constexpr int NT = 256;                 // threads
    constexpr int RW = IT_TX + 16;          // 80 staged columns (halo 8 each side, 16-byte aligned)
    constexpr int RH = TY + 2 * M_;      // staged rows
    constexpr int CH = RH * RW;             // floats per plane box
    constexpr int NC = IT_TX + 2 * M_;      // columns the vertical pass must produce
    constexpr int NW = NT / 32;             // warps
    extern __shared__ __align__(128) float box[];   // [5][RH][RW]
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // 1-D grid with the pair index fastest: CTAs that run at the same time work on the SAME tile of consecutive
    // pairs, and R1 of pair p is R0 of pair p+1 (sequence mode), so every R plane is fetched from HBM once and
    // served to its second reader from L2
    // (the last iteration reads no R: it keeps tile-fastest order, which is better for the M halo reuse)
    // pairs are interleaved in groups of IT_PAIR_GROUP
    const int n_tiles = gridDim.x / a.n_pairs;
    int p, tile;
    if (LAST) {
        p = blockIdx.x / n_tiles;
        tile = blockIdx.x - p * n_tiles;
    } else {
        const int per_group = IT_PAIR_GROUP * n_tiles;
        const int gidx = blockIdx.x / per_group, rem = blockIdx.x - gidx * per_group;
        const int gsize = min(IT_PAIR_GROUP, a.n_pairs - gidx * IT_PAIR_GROUP);     // the last group may be short
        tile = rem / gsize;
        p = gidx * IT_PAIR_GROUP + (rem - tile * gsize);
    }
    const int x0 = (tile % a.tiles_x) * IT_TX, y0 = (tile / a.tiles_x) * TY;
    const int w = a.w, h = a.h, pitch = a.pitch;
    const int plane = (int)a.plane;
    float gk[M_ + 1];                        // Gaussian half kernel (GAUSS only)
#pragma unroll
    for (int i = 0; i <= M_; ++i) gk[i] = GAUSS ? __ldg(a.gk + i) : 0.f;
    auto hsum = [&](const float (&u)[20], float (&o)[4]) {
        if (GAUSS) hsum_gauss_reg<M_>(u, gk, o);
        else hsum_box<M_>(u, o);
    };

    if (tid == 0) {
        // the issuing thread initialises the barrier and starts the load before the block-wide sync that publishes
        // the barrier to the waiters, so the transfer is already in flight while the other warps arrive
        mbar_init(&bar, 1);
        mbar_expect_tx(&bar, 5 * CH * (uint32_t)sizeof(float));
        tma_load_3d(box, &tmap, x0 - 8, y0 - M_, p * 5, &bar);
        // R0 (this tile) and R1 (this tile displaced by the flow) are read ~10 us from now by the per-pixel
        // phase: start their HBM -> L2 transfer now (10 consecutive planes = both frames' expansions)
        if (!LAST) tma_prefetch_3d(&tmapR, x0 - 8, y0 - 8, p * a.pair_stride * 5);
    }
    const bool interior = (x0 - 8 >= 0) && (x0 + IT_TX + 8 <= w) && (y0 - M_ >= 0) && (y0 + TY + M_ <= h);
    __syncthreads();
    mbar_wait(&bar, 0);

    if (!interior) {
        // replicate borders: every out-of-image cell takes the value of the clamped (in-image) cell.  Only the
        // out-of-image cells are visited — first the columns left / right of the image on the in-image rows, then
        // whole rows above / below it (which copy already completed rows) — a few hundred cells per plane, not the
        // whole box: border tiles are 12 % of a 1080p level and up to 40 % of the coarse ones, and walking all
        // 5 x RH x 80 cells with a division each made such a tile cost twice an interior one
        const int xlo = max(0, 8 - x0), xhi = min(RW, w - x0 + 8);          // in-image box columns [xlo, xhi)
        const int ylo = max(0, M_ - y0), yhi = min(RH, h - y0 + M_);        // in-image box rows [ylo, yhi)
        const int ncol = xlo + (RW - xhi), nrow_in = yhi - ylo;
        if (ncol > 0) {
            const int per_plane = nrow_in * ncol;
            for (int idx = tid; idx < 5 * per_plane; idx += NT) {
                const int c = idx / per_plane, rem = idx - c * per_plane;
                const int rr = ylo + rem / ncol, k = rem % ncol;
                const int cc = k < xlo ? k : xhi + (k - xlo);
                float* row = box + c * CH + rr * RW;
                row[cc] = row[k < xlo ? xlo : xhi - 1];
            }
            __syncthreads();
        }
        const int nrow_out = ylo + (RH - yhi);
        if (nrow_out > 0) {
            const int per_plane = nrow_out * (RW / 4);
            for (int idx = tid; idx < 5 * per_plane; idx += NT) {
                const int c = idx / per_plane, rem = idx - c * per_plane;
                const int k = rem / (RW / 4), q = rem - k * (RW / 4);
                const int rr = k < ylo ? k : yhi + (k - ylo);
                float* pl = box + c * CH;
                reinterpret_cast<float4*>(pl + rr * RW)[q] = reinterpret_cast<const float4*>(pl + (k < ylo ? ylo : yhi - 1) * RW)[q];
            }
            __syncthreads();
        }
    }

    // ---- vertical running sums, in place: 15 warp-tasks (plane, 32-column block) ----
    for (int t = warp; t < 15; t += NW) {
        const int c = t / 3, col = (t - 3 * c) * 32 + lane;
        if (col < NC) {
            float* q = box + c * CH + (8 - M_) + col;
            float in[RH];
            float s = 0.f;
#pragma unroll
            for (int j = 0; j <= 2 * M_; ++j) {
                in[j] = q[j * RW];
                s += in[j];
            }
            if (GAUSS) {
                // weighted window: centre tap first, then the symmetric pairs outwards (iter_kernel's expression)
#pragma unroll
                for (int y = 0; y < TY; ++y) {
                    float g = __fmul_rn(in[y + M_], gk[0]);
#pragma unroll
                    for (int i = 1; i <= M_; ++i) g = __fmaf_rn(in[y + M_ - i] + in[y + M_ + i], gk[i], g);
                    q[y * RW] = g;
                    if (y < TY - 1) in[y + 2 * M_ + 1] = q[(y + 2 * M_ + 1) * RW];
                }
                continue;
            }
            // running sums, re-seeded from the window every 8 rows (bounds the float32 drift; the same association
            // as iter_kernel's 8-row segments, so both kernels produce bit-identical sums)
#pragma unroll
            for (int y = 0; y < TY; ++y) {
                q[y * RW] = s;
                if (y < TY - 1) {
                    in[y + 2 * M_ + 1] = q[(y + 2 * M_ + 1) * RW];
                    if (((y + 1) & 7) == 0) {
                        s = 0.f;
#pragma unroll
                        for (int j = 0; j <= 2 * M_; ++j) s += in[y + 1 + j];
                    } else {
                        s += in[y + 2 * M_ + 1] - in[y];
                    }
                }
            }
        }
    }
    __syncthreads();

    if (LAST) {
        // ---- last iteration: horizontal sums of the five planes and the 2x2 solve in registers ----
        // thread = 4 adjacent pixels of one row: no sums are written back to shared memory, no third barrier, and the
        // flow leaves as two 16-byte stores
        const int q4 = tid & 15, rsub = tid >> 4;
        constexpr int ROWS_PER_IT = NT / 16;
        float2* fl = a.flow + (size_t)p * a.flow_stride;
        const float scale = a.scale;
        const bool vec_ok = (a.flow_pitch & 1) == 0 && (reinterpret_cast<uintptr_t>(fl) & 15) == 0;
#pragma unroll 1
        for (int it = 0; it < TY / ROWS_PER_IT; ++it) {
            const int r = it * ROWS_PER_IT + rsub;
            float o[5][4];
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                const float* row = box + c * CH + r * RW + 4 * q4;
                float u[20];
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float4 v = *reinterpret_cast<const float4*>(row + 4 * j);
                    u[4 * j] = v.x; u[4 * j + 1] = v.y; u[4 * j + 2] = v.z; u[4 * j + 3] = v.w;
                }
                hsum(u, o[c]);
                // the weighted filter keeps its half kernel and 20 inputs live: without this fence the compiler hoists
                // the loads of all five planes above the first filter and spills 152 bytes per thread
                if (GAUSS) asm volatile("" ::: "memory");
            }
            const int x = x0 + 4 * q4, y = y0 + r;
            if (y >= h || x >= w) continue;
            float2 f[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float g11 = o[0][k] * scale, g12 = o[1][k] * scale, g22 = o[2][k] * scale, h1 = o[3][k] * scale,
                            h2 = o[4][k] * scale;
                const float idet = __frcp_rn(g11 * g22 - g12 * g12 + 1e-3f);
                f[k] = make_float2((g11 * h2 - g12 * h1) * idet, (g22 * h1 - g12 * h2) * idet);
            }
            float2* dst = fl + (size_t)y * a.flow_pitch + x;
            if (vec_ok && x + 4 <= w) {
                reinterpret_cast<float4*>(dst)[0] = make_float4(f[0].x, f[0].y, f[1].x, f[1].y);
                reinterpret_cast<float4*>(dst)[1] = make_float4(f[2].x, f[2].y, f[3].x, f[3].y);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (x + k < w) dst[k] = f[k];
            }
        }
        return;
    }

    // ---- per pixel: solve, then UpdateMatrices with R1 through shared memory ----
    // (a) every thread turns the sums of its pixels into flow vectors (registers) and the box is free again;
    // (b) ONE TMA load brings the 5 planes of R1 around the tile, displaced by the flow of the tile centre,
    //     into the box; (c) the bilinear gather reads shared memory with immediate offsets (one base address per
    //     pixel, ~30-cycle latency) instead of 20 global loads.  Pixels whose footprint leaves the box (flow
    //     differs from the centre's by more than ~5 px) take the global path; values are identical either way.
    const float* R0 = a.R + (size_t)(p * a.pair_stride) * 5 * a.plane;
    const float* R1 = R0 + 5 * a.plane;
    float* Mout = a.Mout + (size_t)p * 5 * a.plane;
    // keep the pair's M' base as ONE 64-bit register pair: the compiler otherwise carries (kernel argument + 64-bit
    // element offset) and rebuilds every store address with a 4-instruction add / shift chain instead of one
    // IMAD.WIDE.U32 on the 32-bit element offset
    asm volatile("" : "+l"(Mout));
    const bool edge = (x0 < 5) || (y0 < 5) || (x0 + IT_TX > w - 5) || (y0 + TY > h - 5);
    const float scale = a.scale;
    constexpr int PPT = (IT_TX * TY) / NT;
    __shared__ int s_org[2];
    float ffx[PPT], ffy[PPT];
    {
        // (a0) horizontal sums of the five planes + solve for 4 adjacent pixels per task, in registers
        static_assert(TY % 16 == 0, "16 rows per pass");
        const int q4 = tid & 15, rsub = tid >> 4;
        constexpr int NPASS = TY / 16;
        float4 gx[NPASS], gy[NPASS];
#pragma unroll
        for (int it = 0; it < NPASS; ++it) {
            const int r = it * 16 + rsub;
            float o[5][4];
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                const float* row = box + c * CH + r * RW + 4 * q4;
                float u[20];
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float4 v = *reinterpret_cast<const float4*>(row + 4 * j);
                    u[4 * j] = v.x; u[4 * j + 1] = v.y; u[4 * j + 2] = v.z; u[4 * j + 3] = v.w;
                }
                hsum(u, o[c]);
            }
            float fx4[4], fy4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float g11 = o[0][k] * scale, g12 = o[1][k] * scale, g22 = o[2][k] * scale,
                            h1 = o[3][k] * scale, h2 = o[4][k] * scale;
                const float idet = __frcp_rn(g11 * g22 - g12 * g12 + 1e-3f);
                fx4[k] = (g11 * h2 - g12 * h1) * idet;
                fy4[k] = (g22 * h1 - g12 * h2) * idet;
            }
            gx[it] = make_float4(fx4[0], fx4[1], fx4[2], fx4[3]);
            gy[it] = make_float4(fy4[0], fy4[1], fy4[2], fy4[3]);
        }
        __syncthreads();                       // every vertical sum has been consumed: the box is free
        // (a1) the flow vectors through shared memory: [2][TY][64] floats at the start of the box
#pragma unroll
        for (int it = 0; it < NPASS; ++it) {
            const int o4 = (it * 16 + rsub) * IT_TX + 4 * q4;
            *reinterpret_cast<float4*>(box + o4) = gx[it];
            *reinterpret_cast<float4*>(box + IT_TX * TY + o4) = gy[it];
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
        const int idx = j * NT + tid;
        const int cx = idx & 63, r = idx >> 6;
        ffx[j] = box[idx];
        ffy[j] = box[IT_TX * TY + idx];
        if (cx == IT_TX / 2 && r == TY / 2) {
            // box origin: tile origin displaced by the centre pixel's flow, x a multiple of 4
            const float cfx = fminf(fmaxf(ffx[j], -1.0e5f), 1.0e5f), cfy = fminf(fmaxf(ffy[j], -1.0e5f), 1.0e5f);
            s_org[0] = ((x0 + (int)floorf(cfx == cfx ? cfx : 0.f)) & ~3) - 8;
            s_org[1] = y0 + (int)floorf(cfy == cfy ? cfy : 0.f) - M_;
        }
    }
    __syncthreads();                           // all flow vectors read, origin published
    const int bx = s_org[0], by = s_org[1];
    if (tid == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy reads before the async write
        mbar_expect_tx(&bar, 5 * CH * (uint32_t)sizeof(float));
        tma_load_3d(box, &tmapRbox, bx, by, (p * a.pair_stride + 1) * 5, &bar);
    }
    // R0 of the first pixel is requested before waiting for the box, and R0 of pixel j + 1 while pixel j is being
    // worked on: the (L2-prefetched) loads are never waited for
    const int cxp = tid & 63, xp = x0 + cxp;
    const bool col_ok = xp < w;
    auto r0_of = [&](int j) {
        const int y = y0 + ((j * NT + tid) >> 6);
        return (col_ok && y < h) ? load_r0(R0, (unsigned)(y * pitch + xp), (unsigned)plane) : R0Px{0.f, 0.f, 0.f, 0.f, 0.f};
    };
    R0Px cur = r0_of(0);
    mbar_wait(&bar, 1);
#pragma unroll
    for (int j = 0; j < PPT; ++j) {         // fully unrolled: ffx / ffy stay in registers
        const int y = y0 + ((j * NT + tid) >> 6);
        R0Px nxt = cur;
        if (j + 1 < PPT) nxt = r0_of(j + 1);
        if (col_ok && y < h)
            update_matrices_box<RW, RH>(xp, y, w, h, pitch, (unsigned)plane, edge, ffx[j], ffy[j], cur, R1, Mout, box, bx, by);
        cur = nxt;
    }
}

// ------------------------------------------------------------------------------------------------
// taps (tests only): planar pitched -> dense interleaved
// ------------------------------------------------------------------------------------------------
__global__ void tap_planar_kernel(const float* __restrict__ src, int w, int h, int pitch, size_t plane, int nch,
                                  float* __restrict__ dst) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    for (int c = 0; c < nch; ++c) dst[((size_t)y * w + x) * nch + c] = src[c * plane + (size_t)y * pitch + x];
}
__global__ void tap_flow_kernel(const float2* __restrict__ src, int w, int h, int pitch, float2* __restrict__ dst) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    dst[(size_t)y * w + x] = src[(size_t)y * pitch + x];
}

// ------------------------------------------------------------------------------------------------
// host-side orchestration
// ------------------------------------------------------------------------------------------------
template <bool GAUSS, bool LAST>
static int launch_iter(const IterArgs& a, dim3 grid, size_t smem, cudaStream_t s, bool pdl) {
    MAVD_CUDA((ensure_dynamic_smem<iter_kernel<GAUSS, LAST>>(200 * 1024)));
    MAVD_CUDA(launch_chained(pdl, iter_kernel<GAUSS, LAST>, grid, 256, smem, s, a));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

template <int M_, bool LAST, int TY, bool GAUSS>
static int launch_iter_tma(const CUtensorMap& map, const CUtensorMap& mapR, const CUtensorMap& mapRbox, const IterArgs& a,
                           dim3 grid, cudaStream_t s, bool pdl) {
    constexpr size_t smem = sizeof(float) * 5 * (TY + 2 * M_) * (IT_TX + 16);
    MAVD_CUDA((ensure_dynamic_smem<iter_box_tma_kernel<M_, LAST, TY, GAUSS>>(smem)));
    MAVD_CUDA(launch_chained(pdl, iter_box_tma_kernel<M_, LAST, TY, GAUSS>, grid, 256, smem, s, map, mapR, mapRbox, a));
    MAVD_LAUNCHED();
    return MAVD_OK;
}

// 5 <= m <= 8; with small_tiles the caller built `grid` and the descriptors for 64 x 16 tiles
template <bool LAST>
static int launch_iter_tma_m(int m, bool gauss, bool small_tiles, const CUtensorMap& map, const CUtensorMap& mapR,
                             const CUtensorMap& mapRbox, const IterArgs& a, dim3 grid, cudaStream_t s, bool pdl) {
    using Launch = int (*)(const CUtensorMap&, const CUtensorMap&, const CUtensorMap&, const IterArgs&, dim3, cudaStream_t,
                           bool);
#define ITER_TMA_M(TY, GAUSS)                                                                                             \
    { launch_iter_tma<5, LAST, TY, GAUSS>, launch_iter_tma<6, LAST, TY, GAUSS>, launch_iter_tma<7, LAST, TY, GAUSS>,     \
      launch_iter_tma<8, LAST, TY, GAUSS> }
    static const Launch table[2][2][4] = {   // [Gaussian window][64 x 16 tiles][m - 5]
        {ITER_TMA_M(IT_TY, false), ITER_TMA_M(16, false)},
        {ITER_TMA_M(IT_TY, true), ITER_TMA_M(16, true)}};
#undef ITER_TMA_M
    return table[gauss][small_tiles][m - 5](map, mapR, mapRbox, a, grid, s, pdl);
}

int farneback_run(mavd_handle H, const uint8_t* d_frames, int n_pairs, int pair_stride, float* d_flow,
                  cudaStream_t s) {
    const mavd_farneback_params& fp = H->cfg.farneback;
    const int W = H->cfg.width, Hh = H->cfg.height;
    const int n_frames = pair_stride == 1 ? n_pairs + 1 : 2 * n_pairs;
    const bool gauss = (fp.flags & MAVD_FARNEBACK_GAUSSIAN) != 0;
    const int m = fp.winsize / 2;
    const int hx = round_up(m, 4);
    const size_t frame_bytes = (size_t)W * Hh;

    // pyramid images of every coarser level for all frames: two launches
    // pyramid images of levels lo..hi (1 <= lo <= hi) for all frames: two launches
    // programmatic dependent launch: lane 0 = the caller's stream, lane 1 = the side stream (common.cuh: pdl_next)
    auto lane = [&](cudaStream_t st) { return (st == H->s_aux && st != s) ? 1 : 0; };
    pdl_break(H, 0);
    pdl_break(H, 1);
    auto build_pyramid = [&](cudaStream_t st, int lo, int hi) -> int {
        if (H->n_levels <= 1 || lo > hi) return MAVD_OK;
        ProfScope ps(&H->prof, MAVD_PROF_PYRAMID, st);
        const int Wp = round_up(W, 4);
        const bool pyr_staged_env = H->tune.pyr_staged != 0;
        const int word_ok = ((W & 3) == 0 && (reinterpret_cast<uintptr_t>(d_frames) & 3) == 0) ? 1 : 0;
        // descriptor of levels a..b for the generic kernels
        auto make_desc = [&](int a, int b, PyrDesc& d, int& rows) {
            d.n = b - a + 1;
            rows = 0;
            for (int li = a; li <= b; ++li) {
                const Level& L = H->lv[li];
                PyrLevel& P = d.lv[li - a];
                P.w = L.w; P.h = L.h; P.pitch = L.pitch; P.taps = round_up(L.ksz + 1, 4);
                P.xbase = L.xbase; P.xtab = L.xtab; P.ybase = L.ybase; P.ytab = L.ytab;
                P.tmp = L.tmp; P.img = L.img; P.tmp_stride = (size_t)L.h * Wp; P.img_stride = L.plane;
                P.xtabT = L.xtabT;
                P.staged = (pyr_staged_env && L.hspan_max <= PYR_SPAN_MAX && L.hstride_min >= 8) ? 1 : 0;
                P.row0 = rows;
                rows += ceil_div(L.h, 4);
                P.htiles_x = ceil_div(L.w, 64);
            }
        };
        // exact power-of-two levels (leading levels of a pyr_scale 0.5 pyramid): one sweep down the frame does their
        // vertical passes, level 1 and 2 get the vectorised horizontal pass (tuning.pyr_sweep; HalfPyr above)
        int nv = 0, nh = 0;
        if (H->tune.pyr_sweep != 0 && lo == 1 && word_ok) {
            while (nv < VS_MAXLV && 1 + nv <= hi && H->lv[1 + nv].y_half) ++nv;
            while (nh < HP_MAXLV && 1 + nh <= hi && H->lv[1 + nh].x_half) ++nh;
        }
        MAVD_REQUIRE(n_frames <= 65535, MAVD_ERR_UNSUPPORTED, "pyramid: grid too large");
        if (nv > 0) {
            VSweepDesc vd;
            memset(&vd, 0, sizeof(vd));
            for (int l = 0; l < nv; ++l) {
                const Level& L = H->lv[1 + l];
                vd.tmp[l] = L.tmp; vd.tmp_stride[l] = (size_t)L.h * Wp; vd.h[l] = L.h;
                memcpy(vd.w[l], L.ywt, sizeof(float) * VS_MAXT);
            }
            const int words = W / 4, h_top = H->lv[nv].h;
            // bands: enough threads to fill the GPU; each band sweeps 3 steps more than it owns
            int nb = H->tune.pyr_sweep >= 2 ? H->tune.pyr_sweep
                                            : ceil_div(148 * 768, max(1, words * n_frames));
            nb = max(1, min(nb, max(1, h_top / 4)));
            vd.band_rows = ceil_div(h_top, nb);
            nb = ceil_div(h_top, vd.band_rows);
            int tb = 128, waste = 1 << 30;
            for (int cand : {192, 160, 128, 96, 64}) {
                const int wst = ceil_div(words, cand) * cand - words;
                if (wst < waste) { waste = wst; tb = cand; }
            }
            const dim3 g(ceil_div(words, tb), nb, n_frames);
            const bool pdl = pdl_next(H, lane(st));
            // level 1's horizontal pass inside the sweep whenever level 1 is a horizontal decimation too: its vertical
            // sums never go through HBM (C2 pyramid 0.507 -> 0.468 ms on the B200, profiles/README.md).  Level 1 is not
            // one when pyr_scale is close to but not 0.5 and only the height halves exactly, e.g. 640 x 200 at 0.498:
            // level 1 is 319 x 100.
            const bool h1_fused = nh >= 1;
            if (h1_fused) {
                const Level& L1 = H->lv[1];
                vd.img1 = L1.img; vd.img1_stride = L1.plane; vd.pitch1 = L1.pitch;
                memcpy(vd.xw1, L1.xwt, sizeof(vd.xw1));
            }
#define VS_ARGS g, tb, 0, st, d_frames, frame_bytes, W, Hh, Wp, vd
            switch (nv * 2 + (h1_fused ? 1 : 0)) {
                case 2: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<1, false>, VS_ARGS)); break;
                case 3: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<1, true>, VS_ARGS)); break;
                case 4: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<2, false>, VS_ARGS)); break;
                case 5: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<2, true>, VS_ARGS)); break;
                case 6: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<3, false>, VS_ARGS)); break;
                case 7: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<3, true>, VS_ARGS)); break;
                case 8: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<4, false>, VS_ARGS)); break;
                default: MAVD_CUDA(launch_chained(pdl, pyr_vsweep_kernel<4, true>, VS_ARGS)); break;
            }
#undef VS_ARGS
            MAVD_LAUNCHED();
        }
        if (lo + nv <= hi) {
            PyrDesc d;
            int rows = 0;
            make_desc(lo + nv, hi, d, rows);
            MAVD_REQUIRE(rows <= 65535, MAVD_ERR_UNSUPPORTED, "pyramid: grid too large");
            MAVD_CUDA(launch_chained(pdl_next(H, lane(st)), pyr_vfirst_kernel, dim3(ceil_div(W, 256), rows, n_frames), 256, 0, st,
                                     d_frames, frame_bytes, W, Hh, Wp, word_ok, d));
            MAVD_LAUNCHED();
        }
        // level 1 here only when the sweep did not run: level 1 is then not a vertical decimation (e.g. an odd height)
        for (int l = nv >= 1 ? 2 : 1; l <= nh; ++l) {
            const Level& L = H->lv[l];
            HPassW hw;
            memcpy(hw.w, L.xwt, sizeof(hw.w));
            const dim3 g(ceil_div(l <= 2 ? ceil_div(L.w, 4) : L.w, 128), L.h, n_frames);
            MAVD_REQUIRE(L.h <= 65535, MAVD_ERR_UNSUPPORTED, "pyramid: grid too large");
            const bool pdl = pdl_next(H, lane(st));
#define HP_ARGS g, 128, 0, st, (const float*)L.tmp, (size_t)L.h * Wp, W, Wp, L.w, L.img, L.plane, L.pitch, hw
            switch (l) {
                case 1: MAVD_CUDA(launch_chained(pdl, pyr_hpass_kernel<1>, HP_ARGS)); break;
                case 2: MAVD_CUDA(launch_chained(pdl, pyr_hpass_kernel<2>, HP_ARGS)); break;
                case 3: MAVD_CUDA(launch_chained(pdl, pyr_hpass1_kernel<3>, HP_ARGS)); break;
                case 4: MAVD_CUDA(launch_chained(pdl, pyr_hpass1_kernel<4>, HP_ARGS)); break;
                case 5: MAVD_CUDA(launch_chained(pdl, pyr_hpass1_kernel<5>, HP_ARGS)); break;
                default: MAVD_CUDA(launch_chained(pdl, pyr_hpass1_kernel<6>, HP_ARGS)); break;
            }
#undef HP_ARGS
            MAVD_LAUNCHED();
        }
        if (lo + nh <= hi) {
            PyrDesc d;
            int rows = 0;
            make_desc(lo + nh, hi, d, rows);
            MAVD_REQUIRE(rows <= 65535, MAVD_ERR_UNSUPPORTED, "pyramid: grid too large");
            // levels whose outputs are >= 8 source samples apart go through the shared-memory variant: one launch per run
            // of consecutive levels of the same kind (normally two: the fine levels direct, the coarse tail staged)
            for (int a0 = 0; a0 < d.n;) {
                int a1 = a0, hx = 0;
                while (a1 < d.n && d.lv[a1].staged == d.lv[a0].staged) { hx = max(hx, d.lv[a1].htiles_x); ++a1; }
                const int r0 = d.lv[a0].row0, r1 = a1 < d.n ? d.lv[a1].row0 : rows;
                MAVD_CUDA(launch_chained(pdl_next(H, lane(st)), d.lv[a0].staged ? pyr_hsecond_staged_kernel : pyr_hsecond_kernel,
                                         dim3(hx, r1 - r0, n_frames), 256, 0, st, W, Wp, r0, d));
                MAVD_LAUNCHED();
                a0 = a1;
            }
        }
        return MAVD_OK;
    };
    // polynomial expansion of one level for all frames (level 0 reads the u8 frames and blurs on the fly)
    auto expand_level = [&](int li, cudaStream_t st) -> int {
        Level& L = H->lv[li];
        ProfScope ps(&H->prof, MAVD_PROF_POLYEXP, st);
        dim3 g(ceil_div(L.w, PE_TX), ceil_div(L.h, PE_TY), n_frames);
        const int aligned = ((reinterpret_cast<uintptr_t>(d_frames) & 3) == 0 && (W & 3) == 0) ? 1 : 0;
        // TMA-staged tiles: level 0 needs a descriptor of the caller's frames (16-byte aligned rows), built per call
        CUtensorMap tmap_u8;
        bool use_tma = H->tune.polyexp_tma != 0;
        if (use_tma && li == 0)
            use_tma = (W % 16 == 0) && encode_tensor_map_3d(&tmap_u8, true, d_frames, (uint64_t)W, (uint64_t)Hh,
                                                            (uint64_t)n_frames, (uint64_t)W, (uint64_t)W * Hh, PE_BW,
                                                            (uint32_t)(PE_TY + 2 * H->poly.n + 2), 1u);
        else if (use_tma)
            use_tma = L.has_tmap_img;
        const bool pdl = pdl_next(H, lane(st));
#define PE_LAUNCH(N)                                                                                                   \
        do {                                                                                                           \
            if (li == 0 && use_tma)                                                                                    \
                MAVD_CUDA(launch_chained(pdl, polyexp_tma_kernel<true, N>, g, 256, 0, st, tmap_u8, L.w, L.h, L.pitch,   \
                                         H->poly, L.R, L.plane));                                                      \
            else if (li == 0)                                                                                          \
                MAVD_CUDA(launch_chained(pdl, polyexp_kernel<true, N>, g, 256, 0, st, (const void*)d_frames,            \
                                         frame_bytes, L.w, L.h, L.pitch, aligned, H->poly, L.R, L.plane));              \
            else if (use_tma)                                                                                          \
                MAVD_CUDA(launch_chained(pdl, polyexp_tma_kernel<false, N>, g, 256, 0, st, L.tmapImg, L.w, L.h,         \
                                         L.pitch, H->poly, L.R, L.plane));                                             \
            else                                                                                                       \
                MAVD_CUDA(launch_chained(pdl, polyexp_kernel<false, N>, g, 256, 0, st, (const void*)L.img, L.plane,     \
                                         L.w, L.h, L.pitch, 0, H->poly, L.R, L.plane));                                \
        } while (0)
        switch (H->poly.n) {
            case 5: PE_LAUNCH(5); break;
            case 7: PE_LAUNCH(7); break;
            case 8: PE_LAUNCH(8); break;
            default: PE_LAUNCH(0); break;
        }
#undef PE_LAUNCH
        MAVD_LAUNCHED();
        return MAVD_OK;
    };
    // matrices from the upsampled coarser flow, then the iterations of one level
    auto solve_level = [&](int li, cudaStream_t st) -> int {
        Level& L = H->lv[li];
        {
            ProfScope ps(&H->prof, MAVD_PROF_MATRICES, st);
            const bool top = (li == H->n_levels - 1);
            const Level* C = top ? nullptr : &H->lv[li + 1];
            const bool tables = H->tune.mat_coord == 1, no_pow2 = H->tune.mat_coord == 2;
            const double xscale = top ? 1.0 : 1.0 / ((double)L.w / C->w), yscale = top ? 1.0 : 1.0 / ((double)L.h / C->h);
            auto is_pow2 = [](double v) { int e; return v > 0.0 && frexp(v, &e) == 0.5 && e > -20 && e <= 1; };
            const int coord = tables ? MI_COORD_TABLES
                                     : (!no_pow2 && is_pow2(xscale) && is_pow2(yscale)) ? MI_COORD_POW2 : MI_COORD_F64;
            const dim3 g3(n_pairs, ceil_div(L.w, MI_TX), ceil_div(L.h, MI_TY));       // pair index fastest
#define MI_ARGS L.R, L.plane, L.w, L.h, L.pitch, (size_t)pair_stride * 5 * L.plane,                                     \
                top ? nullptr : (const float2*)C->flow, top ? 0 : C->w, top ? 0 : C->h, top ? 0 : C->pitch,             \
                top ? 0 : C->plane, L.fxi0, L.fxa, L.fyi0, L.fya, (float)(1.0 / fp.pyr_scale), L.M[0], xscale, yscale, 1
            const bool pdl = pdl_next(H, lane(st));
            if (coord == MI_COORD_TABLES) MAVD_CUDA(launch_chained(pdl, matrices_init_kernel<MI_COORD_TABLES>, g3, 256, 0, st, MI_ARGS));
            else if (coord == MI_COORD_POW2) MAVD_CUDA(launch_chained(pdl, matrices_init_kernel<MI_COORD_POW2>, g3, 256, 0, st, MI_ARGS));
            else MAVD_CUDA(launch_chained(pdl, matrices_init_kernel<MI_COORD_F64>, g3, 256, 0, st, MI_ARGS));
#undef MI_ARGS
            MAVD_LAUNCHED();
        }
        int cur = 0;
        for (int it = 0; it < fp.iterations; ++it) {
            const bool last = (it == fp.iterations - 1);
            IterArgs a;
            a.Min = L.M[cur];
            a.Mout = L.M[cur ^ 1];
            a.R = L.R;
            a.w = L.w; a.h = L.h; a.pitch = L.pitch; a.plane = L.plane;
            a.m = m; a.hx = hx;
            a.scale = gauss ? 1.f : (float)(1.0 / ((double)fp.winsize * fp.winsize));
            a.pair_stride = pair_stride;
            a.gk = gauss ? H->gauss_win : nullptr;
            if (last) {
                if (li == 0) {
                    a.flow = (float2*)d_flow; a.flow_pitch = W; a.flow_stride = (size_t)W * Hh;
                } else {
                    a.flow = (float2*)L.flow; a.flow_pitch = L.pitch; a.flow_stride = L.plane;
                }
            } else {
                a.flow = nullptr; a.flow_pitch = 0; a.flow_stride = 0;
            }
            dim3 g(ceil_div(L.w, IT_TX), ceil_div(L.h, IT_TY), n_pairs);
            a.n_pairs = n_pairs;
            a.tiles_x = g.x;
            // launches that cannot give every SM its three 64 x 32 tiles (a single pair, the coarse levels) use 64 x 16
            // tiles: twice the CTAs, half the serial work per CTA (tuning.iter_small_tiles)
            const bool small_tiles =
                H->tune.iter_small_tiles != 0 && L.has_tmap16 && (long long)g.x * g.y * g.z <= 3LL * 148;
            const dim3 g1(small_tiles ? g.x * ceil_div(L.h, 16) * g.z : g.x * g.y * g.z);
            const int RW = IT_TX + 2 * hx, RH = IT_TY + 2 * m;
            const size_t smem = sizeof(float) * ((size_t)RH * RW + (size_t)IT_TY * RW + 5 * IT_TX * IT_TY);
            ProfScope ps(&H->prof, li > 0 ? MAVD_PROF_ITER_COARSE : (last ? MAVD_PROF_ITER_FULL_LAST : MAVD_PROF_ITER_FULL), st);
            int rc;
            const bool pdl = pdl_next(H, lane(st));
            if (m >= 5 && m <= 8 && L.has_tmap && !H->force_generic_iter) {
                const CUtensorMap& mM = small_tiles ? L.tmapM16[cur] : L.tmapM[cur];
                const CUtensorMap& mRb = small_tiles ? L.tmapRbox16 : L.tmapRbox;
                rc = last ? launch_iter_tma_m<true>(m, gauss, small_tiles, mM, L.tmapR, mRb, a, g1, st, pdl)
                          : launch_iter_tma_m<false>(m, gauss, small_tiles, mM, L.tmapR, mRb, a, g1, st, pdl);
            }
            else if (gauss) rc = last ? launch_iter<true, true>(a, g, smem, st, pdl) : launch_iter<true, false>(a, g, smem, st, pdl);
            else       rc = last ? launch_iter<false, true>(a, g, smem, st, pdl) : launch_iter<false, false>(a, g, smem, st, pdl);
            if (rc != MAVD_OK) return rc;
            if (!last) cur ^= 1;
        }
        L.last_m = cur;
        return MAVD_OK;
    };

    // The coarse levels (>= 2) are chains of small, latency-bound launches (a 60x34 level is 2 tiles per pair); the
    // expansions of levels 1 and 0 are large and depend only on the frames / pyramid.  Run the coarse chain on a
    // high-priority side stream while the caller's stream does the two big expansions, and join before level 1's
    // matrices need the level-2 flow.  The pyramid goes to the side stream too: level 0's expansion reads only the u8
    // frames.  Stream order as seen by the caller is unchanged.
    const bool fork = H->n_levels >= 3 && H->s_aux != nullptr;
    const int top_level = H->n_levels - 1;
    if (fork) {
        MAVD_CUDA(cudaEventRecord(H->ev_fork, s));
        MAVD_CUDA(cudaStreamWaitEvent(H->s_aux, H->ev_fork, 0));
        pdl_break(H, lane(H->s_aux));
        TRY_RC(build_pyramid(H->s_aux, 1, top_level));
        MAVD_CUDA(cudaEventRecord(H->ev_pyr, H->s_aux));
        for (int li = H->n_levels - 1; li >= 2; --li) {
            TRY_RC(expand_level(li, H->s_aux));
            TRY_RC(solve_level(li, H->s_aux));
        }
        MAVD_CUDA(cudaEventRecord(H->ev_join, H->s_aux));
        TRY_RC(expand_level(0, s));
        MAVD_CUDA(cudaStreamWaitEvent(s, H->ev_pyr, 0));
        pdl_break(H, lane(s));
        TRY_RC(expand_level(1, s));
        MAVD_CUDA(cudaStreamWaitEvent(s, H->ev_join, 0));
        pdl_break(H, lane(s));
        TRY_RC(solve_level(1, s));
        TRY_RC(solve_level(0, s));
    } else {
        TRY_RC(build_pyramid(s, 1, top_level));
        for (int li = H->n_levels - 1; li >= 0; --li) {
            TRY_RC(expand_level(li, s));
            TRY_RC(solve_level(li, s));
        }
    }
    H->last_pairs = n_pairs;
    H->last_stride = pair_stride;
    H->last_flow0 = d_flow;
    H->last_frames = d_frames;
    return MAVD_OK;
}

int farneback_tap(mavd_handle H, int kind, int level, int index, float* d_out, cudaStream_t s) {
    MAVD_REQUIRE(level >= 0 && level < H->n_levels, MAVD_ERR_INVALID, "tap: level %d out of range", level);
    Level& L = H->lv[level];
    dim3 g(ceil_div(L.w, 128), L.h);
    switch (kind) {
        case 0:
            if (level == 0) {
                MAVD_REQUIRE(H->last_frames != nullptr, MAVD_ERR_INVALID, "tap: no farneback call yet");
                pyr0_kernel<<<g, 128, 0, s>>>(H->last_frames + (size_t)index * L.w * L.h, L.w, L.h,
                                              L.img + (size_t)index * L.plane, L.pitch);
                MAVD_LAUNCHED();
            }
            tap_planar_kernel<<<g, 128, 0, s>>>(L.img + (size_t)index * L.plane, L.w, L.h, L.pitch, L.plane, 1, d_out);
            break;
        case 1:
            tap_planar_kernel<<<g, 128, 0, s>>>(L.R + (size_t)index * 5 * L.plane, L.w, L.h, L.pitch, L.plane, 5, d_out);
            break;
        case 2:
            tap_planar_kernel<<<g, 128, 0, s>>>(L.M[L.last_m] + (size_t)index * 5 * L.plane, L.w, L.h, L.pitch,
                                                L.plane, 5, d_out);
            break;
        case 3:
            if (level == 0) {
                MAVD_REQUIRE(H->last_flow0 != nullptr, MAVD_ERR_INVALID, "tap: no farneback call yet");
                tap_flow_kernel<<<g, 128, 0, s>>>((const float2*)H->last_flow0 + (size_t)index * L.w * L.h, L.w, L.h,
                                                  L.w, (float2*)d_out);
            } else {
                tap_flow_kernel<<<g, 128, 0, s>>>((const float2*)L.flow + (size_t)index * L.plane, L.w, L.h, L.pitch,
                                                  (float2*)d_out);
            }
            break;
        default:
            MAVD_REQUIRE(false, MAVD_ERR_INVALID, "tap: unknown kind %d", kind);
    }
    MAVD_LAUNCHED();
    return MAVD_OK;
}

}  // namespace mavd
