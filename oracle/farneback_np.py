"""Stage-wise NumPy restatement of OpenCV's CPU Farneback dense optical flow.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference calls
``cv2.calcOpticalFlowFarneback`` at /root/reference/src/farneback.py:76-80; the
arithmetic itself lives in the third-party ``opencv-python`` wheel (unpinned,
/root/reference/requirements.txt:4; 4.13.0 in this image) whose source
(modules/video/src/optflowgf.cpp) is not vendored.  This module restates the
published algorithm following SURVEY.md Appendix A so that every CUDA kernel
can be checked stage by stage (pyramid image, PolyExp planes, matrices,
per-iteration flow) and not only end to end.  It is pinned against cv2 itself
(tests/test_oracle_farneback.py, tests/golden/farneback_*.npz).

Conventions: images are (H, W) row-major; R and M are (H, W, 5) float32; flow is
(H, W, 2) float32 with the x displacement in channel 0.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np

F32 = np.float32
BORDER = np.array([0.14, 0.14, 0.4472, 0.4472, 0.4472], dtype=np.float32)
OPTFLOW_USE_INITIAL_FLOW = 4
OPTFLOW_FARNEBACK_GAUSSIAN = 256


def cv_round(x: float) -> int:
    """cvRound: round half to even (SSE cvtsd2si default rounding)."""
    return int(np.rint(x))


def level_schedule(width: int, height: int, pyr_scale: float, levels: int,
                   min_size: int = 32) -> List[Tuple[int, float, int, int]]:
    """[(k, scale, w, h)] from the coarsest image down to k=0 (SURVEY §8 a2).

    ``levels = N`` yields up to N+1 images; the cap is ``min_size`` on either side.
    """
    k, s = 0, 1.0
    while k < levels:
        s *= pyr_scale
        if width * s < min_size or height * s < min_size:
            break
        k += 1
    top = k
    out = []
    for k in range(top, -1, -1):
        s = 1.0
        for _ in range(k):
            s *= pyr_scale
        out.append((k, s, cv_round(width * s), cv_round(height * s)))
    return out


def pyramid_blur_params(scale: float) -> Tuple[float, int]:
    sigma = (1.0 / scale - 1.0) * 0.5
    ksz = max(cv_round(sigma * 5) | 1, 3)
    return sigma, ksz


def gaussian_kernel(ksz: int, sigma: float) -> np.ndarray:
    """cv::getGaussianKernel(ksz, sigma, CV_32F)."""
    if sigma <= 0 and ksz in (1, 3, 5, 7):
        tab = {1: [1.0], 3: [0.25, 0.5, 0.25],
               5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
               7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125]}
        return np.array(tab[ksz], dtype=F32)
    if sigma <= 0:
        sigma = ((ksz - 1) * 0.5 - 1) * 0.3 + 0.8
    x = np.arange(ksz, dtype=np.float64) - (ksz - 1) * 0.5
    k = np.exp(-0.5 * x * x / (sigma * sigma))
    k /= k.sum()
    return k.astype(F32)


def _reflect101(idx: np.ndarray, n: int) -> np.ndarray:
    if n == 1:
        return np.zeros_like(idx)
    period = 2 * (n - 1)
    idx = np.mod(idx, period)
    return np.where(idx >= n, period - idx, idx)


def gaussian_blur(img: np.ndarray, ksz: int, sigma: float) -> np.ndarray:
    """cv::GaussianBlur on float32, BORDER_REFLECT_101, separable, f32 accumulate."""
    img = img.astype(F32)
    h, w = img.shape
    k = gaussian_kernel(ksz, sigma)
    r = ksz // 2
    cols = _reflect101(np.arange(-r, w + r), w)
    tmp = np.zeros((h, w), dtype=F32)
    padded = img[:, cols]
    for i in range(ksz):
        tmp += k[i] * padded[:, i:i + w]
    rows = _reflect101(np.arange(-r, h + r), h)
    padded = tmp[rows, :]
    out = np.zeros((h, w), dtype=F32)
    for i in range(ksz):
        out += k[i] * padded[i:i + h, :]
    return out


def _resize_axis_coeffs(src: int, dst: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    inv_scale = dst / src
    scale = 1.0 / inv_scale
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(F32)
    i0 = np.floor(f).astype(np.int64)
    a = (f - i0.astype(F32)).astype(F32)
    lo = i0 < 0
    i0[lo] = 0
    a[lo] = 0
    hi = i0 >= src - 1
    i0[hi] = src - 1
    a[hi] = 0
    i1 = np.minimum(i0 + 1, src - 1)
    return i0, i1, a


def resize_bilinear(src: np.ndarray, w: int, h: int) -> np.ndarray:
    """cv::resize(..., INTER_LINEAR) for float32, 1 or more channels (pixel-centre mapping)."""
    src = src.astype(F32)
    hs, ws = src.shape[:2]
    x0, x1, ax = _resize_axis_coeffs(ws, w)
    y0, y1, ay = _resize_axis_coeffs(hs, h)
    if src.ndim == 3:
        ax_ = ax[None, :, None]
        ay_ = ay[:, None, None]
    else:
        ax_ = ax[None, :]
        ay_ = ay[:, None]
    one = F32(1.0)
    hor = src[:, x0] * (one - ax_) + src[:, x1] * ax_
    out = hor[y0] * (one - ay_) + hor[y1] * ay_
    return out.astype(F32)


def pyramid_image(img_u8: np.ndarray, scale: float, w: int, h: int) -> np.ndarray:
    """I_l = resize(GaussianBlur(f32(img))) always from the full-resolution image (§8 a3)."""
    sigma, ksz = pyramid_blur_params(scale)
    blurred = gaussian_blur(img_u8.astype(F32), ksz, sigma)
    return resize_bilinear(blurred, w, h)


def poly_exp_setup(n: int, sigma: float):
    """FarnebackPrepareGaussian: taps g, xg, xxg (float32, index k=0..n) and ig11, ig03, ig33, ig55."""
    if sigma < np.finfo(np.float32).eps:
        sigma = n * 0.3
    xs = np.arange(-n, n + 1)
    g = np.exp(-(xs * xs) / (2.0 * sigma * sigma)).astype(F32)
    s = 1.0 / float(np.sum(g.astype(np.float64)))
    g = (g.astype(np.float64) * s).astype(F32)
    xg = (xs.astype(F32) * g).astype(F32)
    xxg = ((xs * xs).astype(F32) * g).astype(F32)
    G = np.zeros((6, 6), dtype=np.float64)
    gy = g[:, None]
    gx = g[None, :]
    x_ = xs[None, :].astype(F32)
    y_ = xs[:, None].astype(F32)
    gg = (gy * gx).astype(F32)
    G[0, 0] = float(np.sum(gg.astype(np.float64)))
    G[1, 1] = float(np.sum(((gg * x_) * x_).astype(F32).astype(np.float64)))
    G[3, 3] = float(np.sum(((((gg * x_) * x_) * x_) * x_).astype(F32).astype(np.float64)))
    G[5, 5] = float(np.sum(((((gg * x_) * x_) * y_) * y_).astype(F32).astype(np.float64)))
    G[2, 2] = G[0, 3] = G[0, 4] = G[3, 0] = G[4, 0] = G[1, 1]
    G[4, 4] = G[3, 3]
    G[3, 4] = G[4, 3] = G[5, 5]
    inv = np.linalg.inv(G)
    return (g[n:].copy(), xg[n:].copy(), xxg[n:].copy(),
            float(inv[1, 1]), float(inv[0, 3]), float(inv[3, 3]), float(inv[5, 5]))


def poly_exp(img: np.ndarray, n: int, sigma: float) -> np.ndarray:
    """FarnebackPolyExp: (h, w) f32 -> (h, w, 5) f32 = [r_y, r_x, r_yy, r_xx, r_xy] (§8 a4)."""
    img = img.astype(F32)
    h, w = img.shape
    g, xg, xxg, ig11, ig03, ig33, ig55 = poly_exp_setup(n, sigma)
    rows = np.arange(h)
    t0 = img * g[0]
    t1 = np.zeros_like(img)
    t2 = np.zeros_like(img)
    for k in range(1, n + 1):
        a = img[np.maximum(rows - k, 0)]
        b = img[np.minimum(rows + k, h - 1)]
        t0 = t0 + g[k] * (a + b)
        t1 = t1 + xg[k] * (b - a)
        t2 = t2 + xxg[k] * (a + b)
    cols = np.arange(w)
    D = np.float64
    b1 = (t0 * g[0]).astype(D)
    b3 = (t1 * g[0]).astype(D)
    b5 = (t2 * g[0]).astype(D)
    b2 = np.zeros((h, w), D)
    b4 = np.zeros((h, w), D)
    b6 = np.zeros((h, w), D)
    for k in range(1, n + 1):
        p = np.minimum(cols + k, w - 1)
        m = np.maximum(cols - k, 0)
        tg = (t0[:, p] + t0[:, m]).astype(D)
        b1 += tg * D(g[k])
        b4 += tg * D(xxg[k])
        b2 += ((t0[:, p] - t0[:, m]) * xg[k]).astype(D)
        b3 += ((t1[:, p] + t1[:, m]) * g[k]).astype(D)
        b6 += ((t1[:, p] - t1[:, m]) * xg[k]).astype(D)
        b5 += ((t2[:, p] + t2[:, m]) * g[k]).astype(D)
    R = np.empty((h, w, 5), dtype=F32)
    R[..., 0] = b3 * ig11
    R[..., 1] = b2 * ig11
    R[..., 2] = b1 * ig03 + b5 * ig33
    R[..., 3] = b1 * ig03 + b4 * ig33
    R[..., 4] = b6 * ig55
    return R


def _border_factors(n: int) -> Tuple[np.ndarray, np.ndarray]:
    """Per-index factors from the low edge and from the high edge of one axis of length n (1 elsewhere)."""
    i = np.arange(n)
    lo = np.where(i < 5, BORDER[np.minimum(i, 4)], F32(1)).astype(F32)
    hi = np.where(i >= n - 5, BORDER[np.clip(n - i - 1, 0, 4)], F32(1)).astype(F32)
    return lo, hi


def _border_gate(n: int) -> np.ndarray:
    """cv's (unsigned)(i - 5) >= (unsigned)(n - 10) on one axis.  For n = 8 or 9 the right side wraps to a huge
    unsigned value, so only i in {3, 4} (n = 8) or {4} (n = 9) pass, although every index lies within 5 of an edge."""
    i = np.arange(n, dtype=np.int64)
    return ((i - 5) % 2 ** 32) >= ((n - 10) % 2 ** 32)


def border_scale(w: int, h: int) -> np.ndarray:
    """FarnebackUpdateMatrices' border attenuation (h, w) f32: pixels that pass cv's gate
    (unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10) are scaled by
    ((left * right) * top) * bottom, multiplied in that order in float32; every other pixel by 1."""
    xl, xr = _border_factors(w)
    yt, yb = _border_factors(h)
    sc = ((xl * xr)[None, :] * yt[:, None]).astype(F32) * yb[:, None]
    gate = _border_gate(w)[None, :] | _border_gate(h)[:, None]
    return np.where(gate, sc, F32(1)).astype(F32)


def update_matrices(R0: np.ndarray, R1: np.ndarray, flow: np.ndarray) -> np.ndarray:
    """FarnebackUpdateMatrices (§8 a5): R0, R1 (h,w,5), flow (h,w,2) -> M (h,w,5)."""
    h, w = flow.shape[:2]
    one = F32(1.0)
    dx = flow[..., 0].astype(F32)
    dy = flow[..., 1].astype(F32)
    xs = np.arange(w, dtype=F32)[None, :]
    ys = np.arange(h, dtype=F32)[:, None]
    fx = (xs + dx).astype(F32)
    fy = (ys + dy).astype(F32)
    x1 = np.floor(fx).astype(np.int64)
    y1 = np.floor(fy).astype(np.int64)
    fx = (fx - x1.astype(F32)).astype(F32)
    fy = (fy - y1.astype(F32)).astype(F32)
    inside = (x1 >= 0) & (x1 < w - 1) & (y1 >= 0) & (y1 < h - 1)
    xc = np.clip(x1, 0, max(w - 2, 0))
    yc = np.clip(y1, 0, max(h - 2, 0))
    a00 = (one - fx) * (one - fy)
    a01 = fx * (one - fy)
    a10 = (one - fx) * fy
    a11 = fx * fy
    xr = np.minimum(xc + 1, w - 1)
    yb = np.minimum(yc + 1, h - 1)
    q = (a00[..., None] * R1[yc, xc] + a01[..., None] * R1[yc, xr]
         + a10[..., None] * R1[yb, xc] + a11[..., None] * R1[yb, xr]).astype(F32)
    r2 = np.where(inside, q[..., 0], F32(0))
    r3 = np.where(inside, q[..., 1], F32(0))
    r4 = np.where(inside, (R0[..., 2] + q[..., 2]) * F32(0.5), R0[..., 2])
    r5 = np.where(inside, (R0[..., 3] + q[..., 3]) * F32(0.5), R0[..., 3])
    r6 = np.where(inside, (R0[..., 4] + q[..., 4]) * F32(0.25), R0[..., 4] * F32(0.5))
    r2 = (R0[..., 0] - r2) * F32(0.5)
    r3 = (R0[..., 1] - r3) * F32(0.5)
    r2 = r2 + (r4 * dy + r6 * dx)
    r3 = r3 + (r6 * dy + r5 * dx)
    sc = border_scale(w, h)
    r2, r3, r4, r5, r6 = (v.astype(F32) * sc for v in (r2, r3, r4, r5, r6))
    M = np.empty((h, w, 5), dtype=F32)
    M[..., 0] = r4 * r4 + r6 * r6
    M[..., 1] = (r4 + r5) * r6
    M[..., 2] = r5 * r5 + r6 * r6
    M[..., 3] = r4 * r2 + r6 * r3
    M[..., 4] = r6 * r2 + r5 * r3
    return M


def _box_sum_axis(a: np.ndarray, m: int, axis: int) -> np.ndarray:
    n = a.shape[axis]
    idx = np.clip(np.arange(-m, n + m), 0, n - 1)
    p = np.take(a, idx, axis=axis)
    c = np.cumsum(p, axis=axis, dtype=np.float64)
    zero = np.zeros_like(np.take(c, [0], axis=axis))
    c = np.concatenate([zero, c], axis=axis)
    hi = np.take(c, np.arange(2 * m + 1, n + 2 * m + 1), axis=axis)
    lo = np.take(c, np.arange(0, n), axis=axis)
    return hi - lo


def blur_box(M: np.ndarray, winsize: int) -> np.ndarray:
    """FarnebackUpdateFlow_Blur's blur + 2x2 solve (§8 a6): M (h,w,5) -> flow (h,w,2)."""
    m = winsize // 2
    S = _box_sum_axis(_box_sum_axis(M.astype(np.float64), m, 0), m, 1)
    S *= 1.0 / (winsize * winsize)
    g11, g12, g22, h1, h2 = (S[..., i] for i in range(5))
    idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
    flow = np.empty(M.shape[:2] + (2,), dtype=F32)
    flow[..., 0] = (g11 * h2 - g12 * h1) * idet
    flow[..., 1] = (g22 * h1 - g12 * h2) * idet
    return flow


def gauss_window_kernel(winsize: int) -> np.ndarray:
    """Half kernel k[0..m] of FarnebackUpdateFlow_GaussianBlur (float32, normalised over 2m+1 taps)."""
    m = winsize // 2
    sigma = m * 0.3
    i = np.arange(m + 1, dtype=np.float64)
    k = np.exp(-(i * i) / (2 * sigma * sigma)).astype(F32)
    s = float(k[0]) + 2.0 * float(np.sum(k[1:].astype(np.float64)))
    return (k.astype(np.float64) * (1.0 / s)).astype(F32)


def blur_gauss(M: np.ndarray, winsize: int) -> np.ndarray:
    m = winsize // 2
    k = gauss_window_kernel(winsize)
    h, w = M.shape[:2]
    rows = np.arange(h)
    v = M * k[0]
    for i in range(1, m + 1):
        v = v + (M[np.maximum(rows - i, 0)] + M[np.minimum(rows + i, h - 1)]) * k[i]
    v = v.astype(F32)
    cols = np.arange(w)
    s = v * k[0]
    for i in range(1, m + 1):
        s = s + (v[:, np.maximum(cols - i, 0)] + v[:, np.minimum(cols + i, w - 1)]) * k[i]
    s = s.astype(F32)
    g11, g12, g22, h1, h2 = (s[..., i] for i in range(5))
    idet = F32(1.0) / (g11 * g22 - g12 * g12 + F32(1e-3))
    flow = np.empty((h, w, 2), dtype=F32)
    flow[..., 0] = (g11 * h2 - g12 * h1) * idet
    flow[..., 1] = (g22 * h1 - g12 * h2) * idet
    return flow


def calc_optical_flow_farneback(prev: np.ndarray, nxt: np.ndarray, flow: Optional[np.ndarray],
                                pyr_scale: float, levels: int, winsize: int, iterations: int,
                                poly_n: int, poly_sigma: float, flags: int,
                                tap: Optional[Callable[[str, int, np.ndarray], None]] = None) -> np.ndarray:
    """Same signature as cv2.calcOpticalFlowFarneback (/root/reference/src/farneback.py:76-80).

    ``tap(name, level, array)`` (optional) receives every intermediate:
    'img0','img1','R0','R1','M0' (level entry), and per iteration 'flow<i>' and 'M<i+1>' (the matrices rebuilt from it).
    """
    assert prev.shape == nxt.shape and prev.ndim == 2
    assert pyr_scale < 1
    H, W = prev.shape
    prev_flow = None
    use_init = bool(flags & OPTFLOW_USE_INITIAL_FLOW) and flow is not None
    for k, s, w, h in level_schedule(W, H, pyr_scale, levels):
        if prev_flow is None:
            if use_init:
                cur = (resize_bilinear(flow.astype(F32), w, h) * F32(s)).astype(F32)
            else:
                cur = np.zeros((h, w, 2), dtype=F32)
        else:
            cur = (resize_bilinear(prev_flow, w, h) * F32(1.0 / pyr_scale)).astype(F32)
        R = []
        for j, img in enumerate((prev, nxt)):
            I = pyramid_image(img, s, w, h)
            if tap:
                tap('img%d' % j, k, I)
            R.append(poly_exp(I, poly_n, poly_sigma))
            if tap:
                tap('R%d' % j, k, R[-1])
        M = update_matrices(R[0], R[1], cur)
        if tap:
            tap('M0', k, M)
        for i in range(iterations):
            cur = blur_gauss(M, winsize) if (flags & OPTFLOW_FARNEBACK_GAUSSIAN) else blur_box(M, winsize)
            if tap:
                tap('flow%d' % i, k, cur)
            if i < iterations - 1:
                M = update_matrices(R[0], R[1], cur)
                if tap:
                    tap('M%d' % (i + 1), k, M)
        prev_flow = cur
    return prev_flow
