"""NumPy restatement of OpenCV's sparse feature path: ``cv2.cornerMinEigenVal``, ``cv2.goodFeaturesToTrack`` and
``cv2.calcOpticalFlowPyrLK`` (modules/imgproc/src/corner.cpp, featureselect.cpp; modules/video/src/lkpyramid.cpp).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Pinned against cv2 4.13 stage by stage in tests/test_oracle_lk.py.

What cv2 4.13 does, as pinned:
- Sobel derivatives (gradient size 3) in float32, scaled by 1/(4 * blockSize * 255).  dx is the column filter
  fma(s[y-1] + s[y+1], k, 2k * s[y]) over the exact integer row differences.  dy's row filter [k, 2k, k] is a chain of
  fused multiply-adds for the columns its vector loop covers (x < 32 * floor(W / 32)) and separately rounded products
  and sums for the columns after them; the column difference is one float32 subtraction.
- The products dx*dx, dx*dy, dy*dy are float32; the unnormalised block sum runs in float64 in cv2's order (running
  sums along each row, then down each column) and is rounded to float32 (even block sizes anchor at blockSize // 2).  lambda = (a + c) - sqrt((a - c)^2 + b^2), every operation
  rounded to float32, with a = sum dx^2 / 2, b = sum dx dy, c = sum dy^2 / 2.
- Borders are REFLECT_101 everywhere (the block sum reflects the products' image).
- The quality threshold is compared in float32 (THRESH_TOZERO keeps values strictly above it).

The tracker keeps cv2's fixed-point window sampling exactly; only its float32 accumulation of the gradient matrix and
of the mismatch vector is replaced by exact integer sums, so positions agree with cv2 to the rounding of those sums.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import numpy as np

F32 = np.float32
FLT_EPSILON = float(np.finfo(np.float32).eps)
TERM_COUNT, TERM_EPS = 1, 2
OPTFLOW_LK_GET_MIN_EIGENVALS = 8
SOBEL_VECTOR_COLS = 32   # columns per vector step of cv2's u8 -> f32 row filter (fused multiply-adds inside)


def reflect101(i: np.ndarray, n: int) -> np.ndarray:
    """cv::borderInterpolate(i, n, BORDER_REFLECT_101), repeated until the index lands inside."""
    i = np.asarray(i, np.int64).copy()
    if n == 1:
        return np.zeros_like(i)
    while True:
        bad = (i < 0) | (i >= n)
        if not bad.any():
            return i
        i = np.where(i < 0, -i, i)
        i = np.where(i >= n, 2 * n - 2 - i, i)


def _fma32(a, b, c) -> np.ndarray:
    """float32 fused multiply-add: the float32 product is exact in float64, the sum is rounded once (the operands here
    never span enough exponents for the float64 sum to round)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)


def sobel(img: np.ndarray, block_size: int) -> Tuple[np.ndarray, np.ndarray]:
    """cv2.Sobel(img, CV_32F, 1, 0 / 0, 1, ksize=3, scale=1/(4*block_size*255), BORDER_REFLECT_101) as cv2 4.13
    rounds it."""
    H, W = img.shape
    k1 = F32(1.0 / (4 * block_size * 255.0))
    k0 = F32(2) * k1
    P = img.astype(np.int64)[reflect101(np.arange(-1, H + 1), H)][:, reflect101(np.arange(-1, W + 1), W)]
    r = P[:, 2:] - P[:, :-2]
    dx = _fma32((r[:-2] + r[2:]).astype(F32), k1, r[1:-1].astype(F32) * k0)
    c0, c1, c2 = (P[:, i:i + W].astype(F32) for i in range(3))
    fused = _fma32(c2, k1, _fma32(c1, k0, c0 * k1))
    plain = (c0 * k1 + c1 * k0) + c2 * k1
    n_vec = (W // SOBEL_VECTOR_COLS) * SOBEL_VECTOR_COLS
    row = np.concatenate([fused[:, :n_vec], plain[:, n_vec:]], axis=1)
    dy = row[2:] - row[:-2]
    return dx, dy


def _box_sum(p: np.ndarray, block_size: int) -> np.ndarray:
    """Unnormalised block_size x block_size sum of a float32 image, REFLECT_101, anchor block_size // 2, in float64,
    in cv2's order: each row is a running sum s += (new - old) from the row's left border (direct sums for block sizes
    3 and 5), then each column a running sum down the rows (SUM + new, rounded to float32, then - old)."""
    H, W = p.shape
    k = block_size
    a = k // 2
    q = p.astype(np.float64)[:, reflect101(np.arange(-a, W - a + k - 1), W)]
    if k in (3, 5):
        rows = q[:, 0:W].copy()
        for i in range(1, k):
            rows = rows + q[:, i:i + W]
    else:
        rows = np.empty((H, W), np.float64)
        s = q[:, 0].copy()
        for i in range(1, k):
            s = s + q[:, i]
        rows[:, 0] = s
        for x in range(1, W):
            s = s + (q[:, x + k - 1] - q[:, x - 1])
            rows[:, x] = s
    rows = rows[reflect101(np.arange(-a, H - a + k - 1), H)]
    out = np.empty((H, W), np.float64)
    acc = np.zeros(W, np.float64)
    for i in range(k - 1):
        acc = acc + rows[i]
    for y in range(H):
        s0 = acc + rows[y + k - 1]
        out[y] = s0
        acc = s0 - rows[y]
    return out


def corner_min_eig_val(img: np.ndarray, block_size: int = 3) -> np.ndarray:
    """cv2.cornerMinEigenVal(img, block_size, 3) on a uint8 (H, W) image, bit for bit."""
    dx, dy = sobel(img, block_size)
    sxx = _box_sum(dx * dx, block_size).astype(F32)
    sxy = _box_sum(dx * dy, block_size).astype(F32)
    syy = _box_sum(dy * dy, block_size).astype(F32)
    a = sxx * F32(0.5)
    c = syy * F32(0.5)
    t = a - c
    return ((a + c) - np.sqrt(sxy * sxy + t * t)).astype(F32)


def good_features_to_track(img: np.ndarray, max_corners: int, quality_level: float, min_distance: float,
                           mask: Optional[np.ndarray] = None, block_size: int = 3,
                           eig: Optional[np.ndarray] = None) -> Tuple[np.ndarray, int]:
    """cv2.goodFeaturesToTrack without a corner limit: returns ((N, 2) float32 (x, y) in cv2's order, N).  cv2 with
    maxCorners = k > 0 returns the first k rows; maxCorners <= 0 returns them all."""
    H, W = img.shape
    if eig is None:
        eig = corner_min_eig_val(img, block_size)
    inside = eig if mask is None else eig[mask != 0]
    max_val = float(inside.max()) if inside.size else 0.0
    thr = F32(max_val * quality_level)
    e = np.where(eig > thr, eig, F32(0))
    pad = np.pad(e, 1, constant_values=-np.inf)   # only interior pixels are candidates: the border value is moot
    dil = np.max(np.stack([pad[dy:dy + H, dx:dx + W] for dy in range(3) for dx in range(3)]), axis=0)
    cand = (e != 0) & (e == dil)
    cand[0, :] = cand[-1, :] = False
    cand[:, 0] = cand[:, -1] = False
    if mask is not None:
        cand &= mask != 0
    ys, xs = np.nonzero(cand)
    vals = e[ys, xs]
    pos = ys.astype(np.int64) * W + xs
    order = np.lexsort((-pos, -vals.astype(np.float64)))   # value descending, then later raster position first
    ys, xs = ys[order], xs[order]
    if min_distance >= 1 and len(ys):
        keep = []
        md2 = float(min_distance) * float(min_distance)
        cell = max(1, int(math.ceil(min_distance)))
        grid: dict = {}
        for y, x in zip(ys.tolist(), xs.tolist()):
            cx, cy = x // cell, y // cell
            ok = True
            for gy in (cy - 1, cy, cy + 1):
                for gx in (cx - 1, cx, cx + 1):
                    for (px, py) in grid.get((gx, gy), ()):
                        if (x - px) * (x - px) + (y - py) * (y - py) < md2:
                            ok = False
                            break
                    if not ok:
                        break
                if not ok:
                    break
            if ok:
                grid.setdefault((cx, cy), []).append((x, y))
                keep.append((x, y))
        pts = np.array(keep, np.float32).reshape(-1, 2)
    else:
        pts = np.stack([xs, ys], axis=1).astype(np.float32).reshape(-1, 2)
    return pts, len(pts)


# ---------------------------------------------------------------------------------------------------------------------
# pyramidal Lucas-Kanade

def pyr_down(img: np.ndarray) -> np.ndarray:
    """cv2.pyrDown on uint8: 5-tap [1 4 6 4 1] / 16 each way, REFLECT_101, rounded; size ((w + 1) / 2, (h + 1) / 2)."""
    H, W = img.shape
    h2, w2 = (H + 1) // 2, (W + 1) // 2
    k = np.array([1, 4, 6, 4, 1], np.int64)
    src = img.astype(np.int64)
    cols = reflect101(2 * np.arange(w2)[:, None] + np.arange(-2, 3)[None, :], W)
    rowsum = (src[:, cols] * k).sum(-1)
    rows = reflect101(2 * np.arange(h2)[:, None] + np.arange(-2, 3)[None, :], H)
    tot = (rowsum[rows] * k[None, :, None]).sum(1)
    return ((tot + 128) >> 8).astype(np.uint8)


def scharr_deriv(img: np.ndarray) -> np.ndarray:
    """lkpyramid.cpp calcSharrDeriv: (H, W, 2) int16 (Ix, Iy), 3-10-3 smoothing, REFLECT_101 inside the image."""
    H, W = img.shape
    P = img.astype(np.int32)[reflect101(np.arange(-1, H + 1), H)][:, reflect101(np.arange(-1, W + 1), W)]
    t0 = (P[:-2] + P[2:]) * 3 + P[1:-1] * 10
    t1 = P[2:] - P[:-2]
    ix = t0[:, 2:] - t0[:, :-2]
    iy = (t1[:, 2:] + t1[:, :-2]) * 3 + t1[:, 1:-1] * 10
    return np.stack([ix, iy], -1).astype(np.int16)


def lk_max_level(width: int, height: int, win: Tuple[int, int], max_level: int) -> int:
    """buildOpticalFlowPyramid's level count: a level is kept while the next one is larger than the window."""
    w, h = width, height
    for lvl in range(max_level + 1):
        w, h = (w + 1) // 2, (h + 1) // 2
        if w <= win[0] or h <= win[1]:
            return lvl
    return max_level


def lk_criteria(criteria: Tuple[int, int, float]) -> Tuple[int, float]:
    """(iterations, squared epsilon) as calcOpticalFlowPyrLK normalises the termination criteria."""
    typ, count, eps = criteria
    n = min(max(int(count), 0), 100) if typ & TERM_COUNT else 30
    e = min(max(float(eps), 0.0), 10.0) if typ & TERM_EPS else 0.01
    return n, e * e


def _weights(a: np.ndarray, b: np.ndarray):
    one = F32(1)
    s = F32(1 << 14)
    w00 = np.rint((one - a) * (one - b) * s).astype(np.int64)
    w01 = np.rint(a * (one - b) * s).astype(np.int64)
    w10 = np.rint((one - a) * b * s).astype(np.int64)
    return w00, w01, w10, (1 << 14) - w00 - w01 - w10


def _gather(img: np.ndarray, ix: np.ndarray, iy: np.ndarray, win: Tuple[int, int]) -> np.ndarray:
    """(P, winH + 1, winW + 1) samples of a REFLECT_101-padded image whose window starts at (ix, iy)."""
    H, W = img.shape[:2]
    xs = reflect101(ix[:, None] + np.arange(win[0] + 1)[None, :], W)
    ys = reflect101(iy[:, None] + np.arange(win[1] + 1)[None, :], H)
    return img[ys[:, :, None], xs[:, None, :]]


def _gather_zero(img: np.ndarray, ix: np.ndarray, iy: np.ndarray, win: Tuple[int, int]) -> np.ndarray:
    """The same with zeros outside the image (the derivatives' BORDER_CONSTANT)."""
    H, W = img.shape[:2]
    xs = ix[:, None] + np.arange(win[0] + 1)[None, :]
    ys = iy[:, None] + np.arange(win[1] + 1)[None, :]
    okx, oky = (xs >= 0) & (xs < W), (ys >= 0) & (ys < H)
    v = img[np.clip(ys, 0, H - 1)[:, :, None], np.clip(xs, 0, W - 1)[:, None, :]]
    ok = oky[:, :, None] & okx[:, None, :]
    return np.where(ok[..., None] if v.ndim == 4 else ok, v, 0)


def _interp(s: np.ndarray, w, bits: int) -> np.ndarray:
    w00, w01, w10, w11 = (x[:, None, None] for x in w)
    v = s[:, :-1, :-1] * w00 + s[:, :-1, 1:] * w01 + s[:, 1:, :-1] * w10 + s[:, 1:, 1:] * w11
    return (v + (1 << (bits - 1))) >> bits


def calc_optical_flow_pyr_lk(prev: np.ndarray, nxt: np.ndarray, prev_pts: np.ndarray, win=(21, 21), max_level=3,
                             criteria=(TERM_COUNT | TERM_EPS, 30, 0.01), flags=0, min_eig_threshold=1e-4):
    """cv2.calcOpticalFlowPyrLK(prev, next, prevPts, None, winSize, maxLevel, criteria, flags, minEigThreshold) on
    uint8 frames.  Returns ((N, 2) float32 next points, (N,) uint8 status, (N,) float32 err).  Non-finite points get
    status 0 and err 0 (cv2 leaves them undefined)."""
    pts = np.asarray(prev_pts, np.float32).reshape(-1, 2)
    N = len(pts)
    win = (int(win[0]), int(win[1]))
    H, W = prev.shape
    L = lk_max_level(W, H, win, max_level)
    iters, eps2 = lk_criteria(criteria)
    pyr_i, pyr_j = [prev], [nxt]
    for _ in range(L):
        pyr_i.append(pyr_down(pyr_i[-1]))
        pyr_j.append(pyr_down(pyr_j[-1]))
    finite = np.isfinite(pts).all(1)
    status = finite.astype(np.uint8)
    err = np.zeros(N, np.float32)
    nextp = np.where(finite[:, None], pts, F32(0)).astype(np.float32)
    half = np.array([(win[0] - 1) * 0.5, (win[1] - 1) * 0.5], np.float32)
    area = win[0] * win[1]
    min_eig_t = F32(min_eig_threshold)
    base = np.where(finite[:, None], pts, F32(0)).astype(np.float32)
    for lvl in range(L, -1, -1):
        I, J = pyr_i[lvl], pyr_j[lvl]
        D = scharr_deriv(I).astype(np.int64)
        h, w = I.shape
        pp = base * F32(1.0 / (1 << lvl))
        npt = pp.copy() if lvl == L else nextp * F32(2)
        nextp = npt.copy()
        p0 = pp - half
        ip = np.floor(p0).astype(np.int64)
        live = finite.copy()
        oob = (ip[:, 0] < -win[0]) | (ip[:, 0] >= w) | (ip[:, 1] < -win[1]) | (ip[:, 1] >= h)
        if lvl == 0:
            status[oob & live] = 0
            err[oob & live] = 0
        live &= ~oob
        idx = np.nonzero(live)[0]
        if len(idx) == 0:
            continue
        fr = (p0[idx] - ip[idx].astype(np.float32)).astype(np.float32)
        wts = _weights(fr[:, 0], fr[:, 1])
        Iw = _interp(_gather(I, ip[idx, 0], ip[idx, 1], win).astype(np.int64), wts, 14 - 5)
        Dg = _gather_zero(D, ip[idx, 0], ip[idx, 1], win)
        Ix = _interp(Dg[..., 0], wts, 14)
        Iy = _interp(Dg[..., 1], wts, 14)
        sc = F32(1.0 / (1 << 20))
        A11 = (Ix * Ix).sum((1, 2)).astype(np.float32) * sc
        A12 = (Ix * Iy).sum((1, 2)).astype(np.float32) * sc
        A22 = (Iy * Iy).sum((1, 2)).astype(np.float32) * sc
        Dt = A11 * A22 - A12 * A12
        t = A11 - A22
        min_eig = (A22 + A11 - np.sqrt(t * t + F32(4) * A12 * A12)) / F32(2 * area)
        if flags & OPTFLOW_LK_GET_MIN_EIGENVALS:
            err[idx] = min_eig
        bad = (min_eig < min_eig_t) | (Dt < F32(FLT_EPSILON))
        if lvl == 0:
            status[idx[bad]] = 0
        keep = ~bad
        idx, Iw, Ix, Iy = idx[keep], Iw[keep], Ix[keep], Iy[keep]
        A11, A12, A22 = A11[keep], A12[keep], A22[keep]
        Dinv = F32(1) / Dt[keep]
        cur = (npt[idx] - half).astype(np.float32)
        prev_d = np.zeros_like(cur)
        active = np.ones(len(idx), bool)
        for j in range(iters):
            a_idx = np.nonzero(active)[0]
            if len(a_idx) == 0:
                break
            inp = np.floor(cur[a_idx]).astype(np.int64)
            oob = (inp[:, 0] < -win[0]) | (inp[:, 0] >= w) | (inp[:, 1] < -win[1]) | (inp[:, 1] >= h)
            if lvl == 0:
                status[idx[a_idx[oob]]] = 0
            active[a_idx[oob]] = False
            a_idx, inp = a_idx[~oob], inp[~oob]
            if len(a_idx) == 0:
                break
            fr = (cur[a_idx] - inp.astype(np.float32)).astype(np.float32)
            wts = _weights(fr[:, 0], fr[:, 1])
            Jw = _interp(_gather(J, inp[:, 0], inp[:, 1], win).astype(np.int64), wts, 14 - 5)
            diff = Jw - Iw[a_idx]
            b1 = (diff * Ix[a_idx]).sum((1, 2)).astype(np.float32) * sc
            b2 = (diff * Iy[a_idx]).sum((1, 2)).astype(np.float32) * sc
            dx = (A12[a_idx] * b2 - A22[a_idx] * b1) * Dinv[a_idx]
            dy = (A12[a_idx] * b1 - A11[a_idx] * b2) * Dinv[a_idx]
            delta = np.stack([dx, dy], 1).astype(np.float32)
            cur[a_idx] = cur[a_idx] + delta
            nextp[idx[a_idx]] = cur[a_idx] + half
            small = delta[:, 0].astype(np.float64) ** 2 + delta[:, 1].astype(np.float64) ** 2 <= eps2
            s = prev_d[a_idx] + delta
            ad = np.abs(s).astype(np.float64)   # cv2 compares the float32 sums with the double 0.01
            osc = (j > 0) & (ad[:, 0] < 0.01) & (ad[:, 1] < 0.01) & ~small
            o = a_idx[osc]
            nextp[idx[o]] = nextp[idx[o]] - delta[osc] * F32(0.5)
            active[a_idx[small | osc]] = False
            prev_d[a_idx] = delta
        if lvl == 0 and not flags & OPTFLOW_LK_GET_MIN_EIGENVALS:
            e_idx = idx[status[idx] == 1]
            if len(e_idx):
                q = (nextp[e_idx] - half).astype(np.float32)
                iq = np.floor(q).astype(np.int64)
                oob = (iq[:, 0] < -win[0]) | (iq[:, 0] >= w) | (iq[:, 1] < -win[1]) | (iq[:, 1] >= h)
                status[e_idx[oob]] = 0
                e_idx, q, iq = e_idx[~oob], q[~oob], iq[~oob]
                if len(e_idx):
                    fr = (q - iq.astype(np.float32)).astype(np.float32)
                    wts = _weights(fr[:, 0], fr[:, 1])
                    Jw = _interp(_gather(J, iq[:, 0], iq[:, 1], win).astype(np.int64), wts, 14 - 5)
                    pos = np.searchsorted(idx, e_idx)
                    tot = np.abs(Jw - Iw[pos]).sum((1, 2))
                    err[e_idx] = tot.astype(np.float32) / F32(32 * area)
    nextp[~finite] = pts[~finite]
    return nextp, status, err
