"""8-connected component labelling oracle with canonical (raster first appearance) label numbers.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference has no labelling
stage (SURVEY.md D3/a17) — parity for labels is "unpinned by the reference".
The oracle of record is any correct 8-connected labelling after
canonicalisation; three independent ones are provided and cross-checked in
tests/test_oracle_detect.py: a pure-Python flood fill (small inputs),
scipy.ndimage.label and cv2.connectedComponentsWithStats.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np


def canonicalise(labels: np.ndarray) -> np.ndarray:
    """Renumber labels 1..n in order of first appearance in a raster scan; 0 stays background."""
    flat = labels.ravel()
    fg = np.flatnonzero(flat)
    out = np.zeros(flat.shape, np.int32)
    if fg.size:
        vals, first = np.unique(flat[fg], return_index=True)
        order = np.argsort(first, kind='stable')
        lut = np.zeros(int(vals.max()) + 1, np.int32)
        lut[vals[order]] = np.arange(1, vals.size + 1, dtype=np.int32)
        out[fg] = lut[flat[fg]]
    return out.reshape(labels.shape)


def stats_from_labels(labels: np.ndarray) -> np.ndarray:
    """(n, 5) int32 rows [left, top, width, height, area] for labels 1..n."""
    n = int(labels.max())
    ys, xs = np.nonzero(labels)
    lab = labels[ys, xs].astype(np.int64) - 1
    # one pass over the foreground for all labels at once: a full-HD noise mask has thousands of components, and a
    # pass per label over all of its pixels took minutes
    x0 = np.full(n, np.iinfo(np.int64).max)
    y0 = np.full(n, np.iinfo(np.int64).max)
    x1 = np.full(n, -1, np.int64)
    y1 = np.full(n, -1, np.int64)
    np.minimum.at(x0, lab, xs)
    np.minimum.at(y0, lab, ys)
    np.maximum.at(x1, lab, xs)
    np.maximum.at(y1, lab, ys)
    area = np.bincount(lab, minlength=n)
    return np.stack([x0, y0, x1 - x0 + 1, y1 - y0 + 1, area], axis=1).astype(np.int32).reshape(n, 5)


def label_floodfill(mask: np.ndarray) -> np.ndarray:
    """Pure-Python reference for small masks; labels are canonical by construction."""
    h, w = mask.shape
    lab = np.zeros((h, w), np.int32)
    cur = 0
    for y in range(h):
        for x in range(w):
            if mask[y, x] and lab[y, x] == 0:
                cur += 1
                stack = [(y, x)]
                lab[y, x] = cur
                while stack:
                    cy, cx = stack.pop()
                    for dy in (-1, 0, 1):
                        for dx in (-1, 0, 1):
                            ny, nx = cy + dy, cx + dx
                            if 0 <= ny < h and 0 <= nx < w and mask[ny, nx] and lab[ny, nx] == 0:
                                lab[ny, nx] = cur
                                stack.append((ny, nx))
    return lab


def label_scipy(mask: np.ndarray) -> np.ndarray:
    from scipy import ndimage
    lab, _ = ndimage.label(mask != 0, structure=np.ones((3, 3), np.int32))
    return canonicalise(lab.astype(np.int32))


def label_cv2(mask: np.ndarray) -> np.ndarray:
    import cv2
    _, lab, _, _ = cv2.connectedComponentsWithStats((mask != 0).astype(np.uint8), connectivity=8,
                                                    ltype=cv2.CV_32S)
    return canonicalise(lab)


def label(mask: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    lab = label_scipy(mask)
    return lab, stats_from_labels(lab)
