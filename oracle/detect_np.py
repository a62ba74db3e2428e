"""NumPy restatement of the reference's derotation / FoE / residual / mask / metric stages.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Each function cites the reference
lines it follows; tests/golden/make_golden.py checks these restatements against
the reference modules themselves (imported from /root/reference with stub
dependencies) and commits the resulting vectors.

Parameters.  `intersections`, `ransac`, `foe_dense`, `masks` and `frame_pipeline` take keyword parameters named after
the fields of mavd_detect_params (include/mavd.h).  Their defaults are the reference's constants, and a non-default
value is the reference's expression with that value written in place of the literal.  Pass them as Python floats,
never as np.float64: NumPy follows NEP 50, so a Python float combined with a float32 array is taken as float32
(`np.array([2.4], np.float32) < 2.4` is False, `0.5 + 7.7 / mag` stays float32), which is what the reference does on
its float32 frame (frame_index < 1).  An np.float64 scalar would promote that frame to float64 and change what is
computed.  The segmentation metrics (`simple_bounding_box`, `tpr_fpr`) take graded uint8 masks as the reference does.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

N_PAIRS = 1000  # focus_of_expansion.py:65


def derotation_field(w: int, h: int, ang_diff: np.ndarray, dt: float) -> np.ndarray:
    """Rotational flow predicted from IMU angle deltas — detector.py:88-101.  (h, w, 2) float64."""
    omega = np.asarray(ang_diff, dtype=np.float64) / dt
    col = np.arange(w)[None, :].repeat(h, 0)
    row = np.arange(h)[:, None].repeat(w, 1)
    xn = -(col / w - 0.5) * 2.0
    yn = -(row / h - 0.5) * 2.0
    d0 = +omega[0] * xn * yn - omega[1] * xn ** 2 - omega[1] + omega[2] * yn
    d1 = -omega[2] * xn + omega[0] + omega[0] * yn ** 2 - omega[1] * xn * yn
    out = np.stack([d0, d1], axis=-1)
    out[..., 0] *= w * dt / 2
    out[..., 1] *= h * dt / 2
    return out


def derotate(frame_index: int, flow_uv: np.ndarray, ang_diff: np.ndarray, dt: float) -> np.ndarray:
    """detector.py:70-117: passthrough for frame_index < 1, else flow - derotation (float64)."""
    if frame_index < 1:
        return flow_uv
    h, w = flow_uv.shape[:2]
    return flow_uv - derotation_field(w, h, ang_diff, dt)


def draw_sample_indices(h: int, w: int, rng=np.random) -> Tuple[np.ndarray, np.ndarray]:
    """focus_of_expansion.py:69-71: 2000 row draws, then 2000 column draws, legacy global RNG."""
    ry = rng.randint(0, h, 2 * N_PAIRS)
    rx = rng.randint(0, w, 2 * N_PAIRS)
    return ry, rx


def intersections(flow: np.ndarray, ry: np.ndarray, rx: np.ndarray,
                  magnitude_threshold: float = 2.5) -> np.ndarray:
    """focus_of_expansion.py:74-85 + utils.py:183-197, vectorised.  Returns (K, 2) float64."""
    y1, y2 = ry[:N_PAIRS].astype(np.uint32), ry[N_PAIRS:].astype(np.uint32)
    x1, x2 = rx[:N_PAIRS].astype(np.uint32), rx[N_PAIRS:].astype(np.uint32)
    f1 = flow[y1, x1]
    f2 = flow[y2, x2]
    # get_magnitude(flow2) is evaluated in the flow's own dtype (im_helpers.py:150-159)
    keep = ~(np.linalg.norm(f2, axis=-1) < magnitude_threshold)
    # uint32 + float32/float64 promotes to float64 (focus_of_expansion.py:83)
    c1 = np.stack([x1, y1], -1)
    c2 = np.stack([x2, y2], -1)
    p1 = f1 + c1
    p2 = f2 + c2
    xd0 = c1[:, 0] - p1[:, 0]
    xd1 = c2[:, 0] - p2[:, 0]
    yd0 = c1[:, 1] - p1[:, 1]
    yd1 = c2[:, 1] - p2[:, 1]
    div = xd0 * yd1 - xd1 * yd0
    d0 = c1[:, 0] * p1[:, 1] - c1[:, 1] * p1[:, 0]
    d1 = c2[:, 0] * p2[:, 1] - c2[:, 1] * p2[:, 0]
    ok = keep & (div != 0)
    with np.errstate(divide='ignore', invalid='ignore'):
        ex = (d0 * xd1 - d1 * xd0) / div
        ey = (d0 * yd1 - d1 * yd0) / div
    E = np.zeros((N_PAIRS, 2), np.float64)
    E[ok, 0] = ex[ok]
    E[ok, 1] = ey[ok]
    return E[E[:, 0] != 0.0]


def ransac(E: np.ndarray, ransac_threshold: float = 30.0) -> Tuple[float, float]:
    """focus_of_expansion.py:32-54: score = #within threshold - 1, first strict maximum wins."""
    if E.shape[0] == 0:
        return (0.0, 0.0)
    best, opt = (0.0, 0.0), 0
    for i in range(E.shape[0]):
        d = np.linalg.norm(E - E[i], axis=-1)
        score = int(np.count_nonzero(d < ransac_threshold)) - 1
        if score > opt:
            opt = score
            best = (float(E[i, 0]), float(E[i, 1]))
    return best


def foe_dense(flow: np.ndarray, ry: np.ndarray, rx: np.ndarray, magnitude_threshold: float = 2.5,
              ransac_threshold: float = 30.0) -> Tuple[float, float]:
    return ransac(intersections(flow, ry, rx, magnitude_threshold), ransac_threshold)


def get_phi(flow: np.ndarray, foe: Tuple[float, float], cr_arccos_f32: bool = False) -> np.ndarray:
    """focus_of_expansion.py:150-184: angle [deg] between flow and the ray from the FoE, flow's dtype.

    cr_arccos_f32 (float32 flows only, i.e. frame 0): evaluate arccos correctly rounded (through float64) instead
    of with NumPy's float32 loop.  Every other float32 operation of this function is a single IEEE operation and
    therefore reproducible; NumPy's float32 arccos is NOT correctly rounded and depends on the CPU dispatch
    (AVX-512 SVML here: 35 % of the arguments 1 ulp off, 0.05 % 2 ulp off, measured on 2e7 values), so the reference
    itself is only defined up to those ulps on the float32 frame.  The CUDA path computes the correctly rounded value."""
    h, w = flow.shape[:2]
    d2 = np.zeros_like(flow)
    d2[..., 0] = np.arange(w)[None, :] - foe[0]
    d2[..., 1] = np.arange(h)[:, None] - foe[1]
    a = np.linalg.norm(flow, axis=-1)
    b = np.linalg.norm(d2, axis=-1)
    norm = np.maximum(np.ones_like(a) * 1e-6, a * b)
    c = (flow[..., 0] * d2[..., 0] + flow[..., 1] * d2[..., 1]) / norm
    c = np.clip(c, -1, 1)
    if cr_arccos_f32 and c.dtype == np.float32:
        with np.errstate(invalid='ignore'):
            ang = np.arccos(c.astype(np.float64)).astype(np.float32)
    else:
        ang = np.arccos(c)
    ang[np.isnan(ang)] = 0
    return np.rad2deg(ang)


def masks(flow_derot: np.ndarray, phi: np.ndarray, sky: np.ndarray, dyn_offset: float = 0.25, dyn_base: float = 0.5,
          dyn_gain: float = 8.0, dyn_min_mag: float = 0.5, fixed_min_mag: float = 1.0,
          fixed_angle: float = 15.0) -> Tuple[np.ndarray, np.ndarray]:
    """processor.py:307,333-341 -> (total_mask, estimate_fixed), both bool.  Defaults: the reference's literals."""
    mag = np.linalg.norm(flow_derot, axis=-1)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = dyn_base + dyn_gain / mag
        amax = phi > (dyn_offset + t)
        amin = phi < (dyn_offset - t)
        total = (mag > dyn_min_mag) * ~sky * np.logical_or(amin, amax)
        fixed = phi * (mag > fixed_min_mag) * ~sky > fixed_angle
    return total, fixed


def simple_bounding_box(img: np.ndarray) -> Tuple[int, int, int, int]:
    """im_helpers.py:55-84 -> (x0, y0, x1, y1) of pixels > 0.1*max, -1 when empty."""
    m = img > 0.1 * np.max(img)
    if m.ndim == 3:
        m = m.any(axis=2)
    rows = np.flatnonzero(m.any(axis=1))
    cols = np.flatnonzero(m.any(axis=0))
    if rows.size == 0:
        return (-1, -1, -1, -1)
    return (int(cols[0]), int(rows[0]), int(cols[-1]), int(rows[-1]))


def metric_counts(gt: np.ndarray, mask: np.ndarray) -> Tuple[int, int, int, int]:
    """The four sums of im_helpers.py:244-252 with img = 255*mask (processor.py:350-351): (positives, negatives,
    true positives, false positives) for a uint8 segmentation gt."""
    img = 255 * mask
    p = np.sum(gt > 127)
    n = np.sum((255 - gt) > 127)
    tp = np.sum((gt * img) > 127)
    fp = np.sum(((255 - gt) * img) > 127)
    return p, n, tp, fp


def tpr_fpr(gt: np.ndarray, mask: np.ndarray) -> Tuple[float, float]:
    """im_helpers.py:244-252 with img = 255*mask (processor.py:350-351)."""
    p, n, tp, fp = metric_counts(gt, mask)
    with np.errstate(divide='ignore', invalid='ignore'):
        return (tp / p, fp / n)


def frame_pipeline(frame_index: int, flow_uv: np.ndarray, ang_diff, dt: float, sky: np.ndarray,
                   ry: np.ndarray, rx: np.ndarray, cr_arccos_f32: bool = False, magnitude_threshold: float = 2.5,
                   ransac_threshold: float = 30.0, **mask_params):
    """processor.py:305-341 for one frame given pre-drawn sample indices.  mask_params: the keywords of masks()."""
    fd = derotate(frame_index, flow_uv, ang_diff, dt)
    foe = foe_dense(fd, ry, rx, magnitude_threshold, ransac_threshold)
    phi = get_phi(fd, foe, cr_arccos_f32)
    total, fixed = masks(fd, phi, sky, **mask_params)
    return fd, foe, phi, total, fixed
