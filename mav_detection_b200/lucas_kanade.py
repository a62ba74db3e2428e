"""LucasKanade with the reference's constructor, and the two cv2 calls of its sparse path on the device.

The body of the reference's sparse tracker (src/lucas_kanade.py:9-63) is unused by
Processor.run_detection (SURVEY.md §2), and its parameters and re-detection policy are not recorded, so `get_features`
still raises.  FocusOfExpansion only reads `old_frame.shape` and `total_num_corners` from it (focus_of_expansion.py:24-27).
The constructor keeps the reference's draw from the global legacy NumPy generator (lucas_kanade.py:32) so that the
random stream seen by get_FOE_dense is unchanged.

`goodFeaturesToTrack` and `calcOpticalFlowPyrLK` are the seams that tracker calls: the cv2 functions with cv2's
argument names, defaults, output shapes and dtypes (and cv2's None when no corner is found), computed by the sparse
kernels (csrc/sparse.cu) on `engine.shared_engine(W, H)`."""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib


class LucasKanade:
    def __init__(self, old_frame: np.ndarray) -> None:
        self.old_frame = old_frame
        self.num_corners = 2000
        self.minimum_num_corners = self.num_corners // 3
        self.total_num_corners = self.num_corners + self.minimum_num_corners
        self.corners = np.zeros((self.total_num_corners, 2), dtype=np.uint)
        self.num_features = 0
        self.features = []
        self.color = np.random.randint(0, 255, (self.total_num_corners, 3))

    def get_features(self, frame: np.ndarray):
        raise NotImplementedError('the sparse Lucas-Kanade tracker is outside the rebuilt hot path (SURVEY.md §2)')


def _gray(image: np.ndarray, name: str) -> np.ndarray:
    a = np.asarray(image)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError('%s must be a (H, W) uint8 image' % name)
    return np.ascontiguousarray(a)


def _engine(img: np.ndarray):
    from . import engine
    return engine.shared_engine(img.shape[1], img.shape[0])


def goodFeaturesToTrack(image: np.ndarray, maxCorners: int, qualityLevel: float, minDistance: float,
                        mask: Optional[np.ndarray] = None, blockSize: int = 3, gradientSize: int = 3,
                        useHarrisDetector: bool = False, k: float = 0.04) -> Optional[np.ndarray]:
    """cv2.goodFeaturesToTrack on the device: (N, 1, 2) float32 corners, or None when there is none."""
    if useHarrisDetector:
        raise ValueError('the Harris detector is not supported')
    img = _gray(image, 'image')
    eng = _engine(img)
    dev = eng.device
    frames = torch.from_numpy(img).to(dev).unsqueeze(0)
    m = None if mask is None else torch.from_numpy(_gray(mask, 'mask')).to(dev)
    if int(gradientSize) != 3:
        raise ValueError('gradientSize must be 3')
    want = int(maxCorners)
    corners, counts = eng.good_features(frames, max(want, 0), qualityLevel, minDistance, blockSize, mask=m)
    n = int(counts[0])
    if want <= 0 and n > 0:      # no limit: ask again with room for every corner
        corners, counts = eng.good_features(frames, n, qualityLevel, minDistance, blockSize, mask=m)
    n = n if want <= 0 else min(n, want)
    if n == 0:
        return None
    return corners[0, :n].cpu().numpy().reshape(n, 1, 2)


def calcOpticalFlowPyrLK(prevImg: np.ndarray, nextImg: np.ndarray, prevPts: np.ndarray, nextPts=None,
                         status=None, err=None, winSize: Tuple[int, int] = (21, 21), maxLevel: int = 3,
                         criteria: Tuple[int, int, float] = (_lib.TERM_COUNT | _lib.TERM_EPS, 30, 0.01),
                         flags: int = 0, minEigThreshold: float = 1e-4):
    """cv2.calcOpticalFlowPyrLK on the device: ((N, 1, 2) float32 next points, (N, 1) uint8 status, (N, 1) float32
    err).  The output arguments are accepted for cv2's signature and ignored, as is an initial flow."""
    a, b = _gray(prevImg, 'prevImg'), _gray(nextImg, 'nextImg')
    if a.shape != b.shape:
        raise ValueError('prevImg and nextImg must have the same size')
    pts = np.ascontiguousarray(np.asarray(prevPts, np.float32).reshape(-1, 2))
    eng = _engine(a)
    dev = eng.device
    frames = torch.from_numpy(np.stack([a, b])).to(dev)
    nxt, st, e = eng.pyr_lk(frames, torch.from_numpy(pts).to(dev).unsqueeze(0), pair_stride=2,
                            win=(int(winSize[0]), int(winSize[1])), max_level=int(maxLevel), criteria=tuple(criteria),
                            flags=int(flags), min_eig_threshold=float(minEigThreshold))
    n = len(pts)
    return (nxt[0].cpu().numpy().reshape(n, 1, 2), st[0].cpu().numpy().reshape(n, 1),
            e[0].cpu().numpy().reshape(n, 1))
