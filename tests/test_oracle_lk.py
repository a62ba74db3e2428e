"""CPU: oracle/lk_np.py against live cv2, stage by stage, and the sparse path's ABI and launch invariants.

The eig image must be cornerMinEigenVal's bits, the corner lists goodFeaturesToTrack's (position, order, count), and the
tracker's status calcOpticalFlowPyrLK's on every point.  Positions and err differ from cv2 only by cv2's float32
accumulation of the window sums (the oracle and the kernels sum exactly); the bars below are the measured spread."""
import ctypes as C
import os
import re

import cv2
import numpy as np
import pytest

from mav_detection_b200 import synth
from oracle import lk_np as lk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'mav_detection_b200', 'csrc')
TC, TE = cv2.TERM_CRITERIA_COUNT, cv2.TERM_CRITERIA_EPS


def frame_pair(W, H, seq=0):
    a, b = synth.make_pair(max(W, 64), max(H, 64), seq=seq)
    return np.ascontiguousarray(a[:H, :W]), np.ascontiguousarray(b[:H, :W])


@pytest.mark.parametrize('W,H', [(8, 8), (33, 17), (95, 64), (640, 480), (1920, 1080)])
@pytest.mark.parametrize('bs', [1, 2, 3, 4, 5, 7, 31])
def test_eig_is_corner_min_eig_val(W, H, bs):
    a, _ = frame_pair(W, H)
    assert np.array_equal(lk.corner_min_eig_val(a, bs).view(np.int32), cv2.cornerMinEigenVal(a, bs, ksize=3).view(np.int32))


def test_eig_on_noise_every_width():
    rng = np.random.default_rng(3)
    for W in range(8, 80, 3):
        a = rng.integers(0, 256, (19, W)).astype(np.uint8)
        for bs in (2, 7):
            assert np.array_equal(lk.corner_min_eig_val(a, bs), cv2.cornerMinEigenVal(a, bs, ksize=3)), (W, bs)


def _cv_corners(a, mc, q, md, bs, mask=None):
    c = cv2.goodFeaturesToTrack(a, mc, q, md, mask=mask, blockSize=bs)
    return None if c is None else c.reshape(-1, 2)


def _check_corners(a, mc, q, md, bs, mask=None, eig=None):
    ref = _cv_corners(a, mc, q, md, bs, mask)
    pts, n = lk.good_features_to_track(a, mc, q, md, mask=mask, block_size=bs, eig=eig)
    got = pts[:mc] if mc > 0 else pts
    if ref is None:
        assert len(got) == 0
    else:
        assert np.array_equal(ref, got), (mc, q, md, bs)


@pytest.mark.parametrize('W,H', [(8, 8), (33, 17), (640, 480)])
@pytest.mark.parametrize('bs', [1, 2, 3, 7, 31])
def test_corners_are_cv2s(W, H, bs):
    a, _ = frame_pair(W, H)
    eig = lk.corner_min_eig_val(a, bs)
    for q in (1e-4, 0.01, 0.3, 1.0):
        for md in (0, 0.5, 1, 7, 7.4, 30):
            for mc in (0, 1, 25, 2000):
                _check_corners(a, mc, q, md, bs, eig=eig)


def test_corners_1080p_and_masks():
    a, _ = frame_pair(1920, 1080)
    _check_corners(a, 2000, 0.01, 7, 7)
    _check_corners(a, 0, 0.01, 7.4, 3)
    rng = np.random.default_rng(1)
    b, _ = frame_pair(640, 480)
    for mask in (rng.integers(0, 2, b.shape).astype(np.uint8) * 255, np.zeros(b.shape, np.uint8)):
        _check_corners(b, 500, 0.01, 5, 3, mask=mask)
    m = np.zeros(b.shape, np.uint8)
    m[100:300, 50:400] = 1
    _check_corners(b, 0, 0.05, 3, 7, mask=m)


def test_constant_frame_has_no_corners():
    z = np.full((64, 64), 77, np.uint8)
    assert cv2.goodFeaturesToTrack(z, 10, 0.01, 3) is None
    assert lk.good_features_to_track(z, 10, 0.01, 3)[1] == 0


def test_pyramid_and_derivatives():
    for W, H in [(8, 8), (33, 17), (640, 480), (101, 77)]:
        a, _ = frame_pair(W, H)
        assert np.array_equal(lk.pyr_down(a), cv2.pyrDown(a))
        assert lk.lk_max_level(W, H, (21, 21), 8) == len(cv2.buildOpticalFlowPyramid(a, (21, 21), 8, withDerivatives=False)[1]) - 1
    assert lk.lk_max_level(80, 60, (21, 21), 5) == 1


def _lk_points(a, W, H, rng):
    p = cv2.goodFeaturesToTrack(a, 300, 0.01, 3)
    p = np.zeros((0, 2), np.float32) if p is None else p.reshape(-1, 2)
    extra = [rng.uniform([-30, -30], [W + 30, H + 30], (100, 2)),
             np.array([[0, 0], [W - 1, H - 1], [-1, 5], [W, 3], [5, H], [-25, -25], [W + 40, 2]], float)]
    return np.concatenate([p] + [e.astype(np.float32) for e in extra]).astype(np.float32)


LK_CASES = [((21, 21), 3, 0, (TC | TE, 30, 0.01), 1e-4), ((15, 15), 2, 8, (TC | TE, 10, 0.03), 1e-4),
            ((3, 3), 0, 0, (TE, 5, 0.01), 0), ((31, 9), 8, 0, (TC, 500, 0), 1e-2), ((63, 63), 3, 8, (TC | TE, 30, 20), 1e-4),
            ((21, 21), 5, 0, (TC, -3, 0), 1e-4), ((15, 15), 4, 0, (0, 0, 0), 1e-2)]


def check_lk(ref, got, win, far=0.0):
    """far: the share of status-1 points allowed further than 0.01 px from cv2 (iterations that diverge)."""
    (n1, s1, e1), (n2, s2, e2) = ref, got
    s1 = s1.ravel()
    assert np.array_equal(s1, s2.ravel())
    ok = s1 == 1
    if not ok.any():
        return
    d = np.abs(n1.reshape(-1, 2) - n2.reshape(-1, 2))[ok].max(1)
    # a 3 x 3 window is too small to pin the solve: cv2's rounded sums can end its iteration elsewhere
    if min(win) > 3:
        assert (d > 0.01).mean() <= far, ((d > 0.01).mean(), d.max())
        # measured: >= 98.9 % on the synthetic pairs, 92 % under 8-40 px shifts (more iterations on coarse levels,
        # each carrying cv2's float32 rounding of the window sums)
        assert (d <= 1e-4).mean() >= 0.9, (d <= 1e-4).mean()
        # err (mean absolute residual, 0..255 intensity units) is sampled where the point ends, so the position residue
        # moves it: measured up to 2.4e-2 (640 x 480, maxLevel 0-8) and 9.3e-3 under 8-40 px shifts
        assert np.abs(e1.ravel() - e2.ravel())[ok][d <= 0.01].max() <= 5e-2


@pytest.mark.parametrize('W,H', [(8, 8), (80, 60), (640, 480), (1920, 1080)])
def test_lk_matches_cv2(W, H):
    a, b = frame_pair(W, H)
    rng = np.random.default_rng(W)
    q = _lk_points(a, W, H, rng)
    for win, ml, fl, cr, me in LK_CASES:
        ref = cv2.calcOpticalFlowPyrLK(a, b, q.reshape(-1, 1, 2), None, winSize=win, maxLevel=ml, criteria=cr, flags=fl,
                                       minEigThreshold=me)
        check_lk(ref, lk.calc_optical_flow_pyr_lk(a, b, q, win, ml, cr, fl, me), win)


def test_lk_large_motion_needs_the_pyramid():
    seq = synth.make_sequence(320, 240, 2, seq=0, with_rotation=True)
    a, b = seq.frames[0], seq.frames[1]
    rng = np.random.default_rng(0)
    for shift in (8, 20, 40):
        c = np.roll(a, (shift // 2, shift), axis=(0, 1))
        q = _lk_points(a, 320, 240, rng)
        for ml in (0, 3):
            ref = cv2.calcOpticalFlowPyrLK(a, c, q.reshape(-1, 1, 2), None, winSize=(21, 21), maxLevel=ml)
            # np.roll wraps the frame: windows across the seam are ill-conditioned and can end far apart
            check_lk(ref, lk.calc_optical_flow_pyr_lk(a, c, q, (21, 21), ml), (21, 21), far=0.01)
    del b


def test_lk_non_finite_points():
    a, b = frame_pair(64, 64)
    q = np.array([[np.nan, 3], [5, np.inf], [10, 10]], np.float32)
    n, s, e = lk.calc_optical_flow_pyr_lk(a, b, q)
    assert list(s[:2]) == [0, 0] and list(e[:2]) == [0, 0]


_CTYPES = {'int32_t': C.c_int32, 'double': C.c_double}


@pytest.mark.parametrize('name,cls', [('mavd_gftt_params', 'GfttParams'), ('mavd_lk_params', 'LkParams')])
def test_param_structs_are_the_header_member_lists(name, cls):
    from mav_detection_b200 import _lib
    src = re.sub(r'/\*.*?\*/', '', open(os.path.join(ROOT, 'include', 'mavd.h')).read(), flags=re.S)
    body = re.search(r'typedef struct %s \{(.*?)\} %s;' % (name, name), src, flags=re.S).group(1)
    members = [(nm.strip(), _CTYPES[t]) for t, names in re.findall(r'(int32_t|double)\s+([^;]+);', body)
               for nm in names.split(',')]
    S = getattr(_lib, cls)
    assert [m for m, _ in members] == [f for f, _ in S._fields_]
    off = 0
    for (m, ct), (f, ft) in zip(members, S._fields_):
        assert ft is ct, m
        off = -(-off // C.sizeof(ct)) * C.sizeof(ct)
        assert getattr(S, m).offset == off, m
        off += C.sizeof(ct)
    assert C.sizeof(S) == -(-off // 8) * 8


def test_sparse_launch_chain_invariants():
    """sparse.cu may not chain a kernel behind an event wait, a memset or a copy (tests/test_launch_chain.py)."""
    lines = open(os.path.join(CSRC, 'sparse.cu')).read().split('\n')
    for i, line in enumerate(lines):
        if 'cudaStreamWaitEvent(' in line and 'MAVD_CUDA' in line:
            assert 'pdl_break' in '\n'.join(lines[i:i + 3]), 'sparse.cu:%d: event wait without pdl_break' % (i + 1)
        if 'cudaMemsetAsync(' in line or 'cudaMemcpyAsync(' in line:
            for k in range(i + 1, min(i + 8, len(lines))):
                if '<<<' in lines[k] or 'return' in lines[k]:
                    break
                if 'launch_chained(' in lines[k]:
                    assert any('pdl_break' in l for l in lines[i:k]), 'sparse.cu:%d: memset / copy, then a chained launch' % (i + 1)
                    break
