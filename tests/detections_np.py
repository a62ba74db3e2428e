"""Detection-table oracle (include/mavd.h: mavd_detection) built on the canonical labelling of oracle/ccl_np.py.

TEST INFRASTRUCTURE: NumPy only, cross-checked against cv2.connectedComponentsWithStats in
tests/test_detections_oracle.py; the GPU tests of tests/test_gpu_detections.py compare the kernels with it."""
from __future__ import annotations

import numpy as np

from oracle.ccl_np import label


# one entry of a frame's detection table, laid out as include/mavd.h: mavd_detection
DETECTION_DTYPE = np.dtype([('label', '<i4'), ('box', '<i4', (4,)), ('area', '<i4'), ('sum_x', '<i8'), ('sum_y', '<i8'),
                            ('flow_sum', '<f8', (2,))])


def detections(mask: np.ndarray, flow_derot: np.ndarray = None, max_det: int = 32) -> np.ndarray:
    """The max_det largest 8-connected components of `mask` (non-zero = foreground), ordered by area descending, then
    canonical label ascending, as (max_det,) DETECTION_DTYPE; entries past the component count are zero.  flow_derot
    (H, W, 2) float64, optional: flow_sum is its sum over each component's pixels (np.add.at), else 0."""
    lab, st = label(mask)
    n = st.shape[0]
    out = np.zeros(max_det, DETECTION_DTYPE)
    if n == 0:
        return out
    ys, xs = np.nonzero(lab)
    li = lab[ys, xs].astype(np.int64) - 1
    area = np.bincount(li, minlength=n)
    sum_x = np.bincount(li, weights=xs, minlength=n).astype(np.int64)   # exact: sums < 2^53
    sum_y = np.bincount(li, weights=ys, minlength=n).astype(np.int64)
    fs = np.zeros((n, 2), np.float64)
    if flow_derot is not None:
        np.add.at(fs, li, flow_derot[ys, xs].astype(np.float64))
    order = np.lexsort((np.arange(n), -area))[:max_det]                  # area desc, then label asc
    k = order.size
    out['label'][:k] = order + 1
    out['box'][:k] = st[order, :4]
    out['area'][:k] = area[order]
    out['sum_x'][:k] = sum_x[order]
    out['sum_y'][:k] = sum_y[order]
    out['flow_sum'][:k] = fs[order]
    return out
