"""CPU: the NumPy Farneback restatement against the committed cv2 vectors and against cv2 itself."""
import glob
import os

import numpy as np
import pytest

from oracle import farneback_np as fb

TOL_MEAN, TOL_MAX = 1e-5, 1e-4   # px; SURVEY.md §7 step 1


def _params(p):
    return (float(p[0]), int(p[1]), int(p[2]), int(p[3]), int(p[4]), float(p[5]), int(p[6]))


@pytest.mark.parametrize('name', ['ref', 'c2', 'gauss', 'odd', 'lvl0'])
def test_oracle_matches_golden_cv2_flow(golden_dir, name):
    g = np.load(os.path.join(golden_dir, 'farneback_%s.npz' % name))
    mine = fb.calc_optical_flow_farneback(g['prev'], g['next'], None, *_params(g['params']))
    epe = np.linalg.norm(mine - g['flow'], axis=-1)
    assert epe.mean() < TOL_MEAN and epe.max() < TOL_MAX


def test_oracle_matches_live_cv2():
    cv2 = pytest.importorskip('cv2')
    from mav_detection_b200 import synth
    a, b = synth.make_pair(200, 144, seq=3)
    for p in [(0.4, 1, 12, 10, 8, 1.2, 0), (0.5, 5, 15, 3, 5, 1.2, 0), (0.5, 2, 9, 2, 7, 1.5, 256)]:
        ref = cv2.calcOpticalFlowFarneback(a, b, None, *p)
        mine = fb.calc_optical_flow_farneback(a, b, None, *p)
        epe = np.linalg.norm(mine - ref, axis=-1)
        assert epe.mean() < TOL_MEAN and epe.max() < TOL_MAX, p


@pytest.mark.parametrize('w,h', [(8, 8), (9, 9), (9, 12), (64, 8), (8, 64), (11, 9), (10, 10), (10, 11),
                                 (16, 16)])
def test_oracle_matches_live_cv2_on_tiny_frames(w, h):
    """Sides of 8 and 9 pixels: cv's border gate (unsigned)(x - 5) >= (unsigned)(w - 10) wraps there and leaves
    most pixels within 5 of an edge unattenuated; 10 and 11 are the first sides where it covers them all."""
    cv2 = pytest.importorskip('cv2')
    from mav_detection_b200 import synth
    a, b = synth.make_pair(64, 64, seq=4)
    a, b = np.ascontiguousarray(a[20:20 + h, 13:13 + w]), np.ascontiguousarray(b[20:20 + h, 13:13 + w])
    for p in [(0.5, 3, 15, 3, 5, 1.2, 0), (0.4, 1, 12, 10, 8, 1.2, 0), (0.5, 2, 21, 2, 7, 1.5, 256)]:
        ref = cv2.calcOpticalFlowFarneback(a, b, None, *p)
        mine = fb.calc_optical_flow_farneback(a, b, None, *p)
        epe = np.linalg.norm(mine - ref, axis=-1)
        assert np.abs(ref).max() > 1e-3, p                  # the border terms carry the result: not vacuous
        assert epe.mean() < TOL_MEAN and epe.max() < TOL_MAX, (p, epe.mean(), epe.max())


def test_border_gate_matches_cv2_unsigned_expression():
    """Which pixels are attenuated, written out for the sides where the unsigned comparison wraps."""
    assert np.flatnonzero(fb._border_gate(8)).tolist() == [3, 4]
    assert np.flatnonzero(fb._border_gate(9)).tolist() == [4]
    assert fb._border_gate(10).all()
    assert np.flatnonzero(~fb._border_gate(11)).tolist() == [5]
    assert np.flatnonzero(~fb._border_gate(64)).tolist() == list(range(5, 59))
    sc = fb.border_scale(8, 8)
    assert sc[0, 0] == 1 and sc[7, 7] == 1                 # outside the gate on both axes
    b = fb.BORDER
    # x = 3 passes the gate: left factor border[3], right factor border[8 - 3 - 1] = border[4]; y = 0 adds border[0]
    # and y = 0 is also 8 - 0 - 1 = 7 >= 5 from the bottom, so no bottom factor
    assert sc[0, 3] == np.float32(np.float32(b[3] * b[4]) * b[0])
    assert sc[3, 3] == np.float32(np.float32(np.float32(b[3] * b[4]) * b[3]) * b[4])


def test_level_schedule_matches_survey():
    # SURVEY §8 a2: C2 1920x1080, levels=5 -> 6 images down to 60x34
    sched = fb.level_schedule(1920, 1080, 0.5, 5)
    assert [(w, h) for _, _, w, h in sched] == [(60, 34), (120, 68), (240, 135), (480, 270), (960, 540), (1920, 1080)]
    # levels capped by the 32-pixel rule at 640x480
    assert len(fb.level_schedule(640, 480, 0.5, 10)) == len(fb.level_schedule(640, 480, 0.5, 3)) == 4
    # reference params: 2 images, 256x192 then 640x480
    assert [(w, h) for _, _, w, h in fb.level_schedule(640, 480, 0.4, 1)] == [(256, 192), (640, 480)]
    assert len(fb.level_schedule(640, 480, 0.5, 0)) == 1


def test_pyramid_blur_params():
    assert fb.pyramid_blur_params(1.0) == (0.0, 3)
    assert fb.pyramid_blur_params(0.5)[1] == 3
    assert fb.pyramid_blur_params(0.25)[1] == 9
    assert fb.pyramid_blur_params(1 / 32)[1] == 79


def test_stage_primitives_against_cv2():
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(0)
    img = (rng.random((77, 123)) * 255).astype(np.float32)
    for ksz, sigma in [(3, 0.0), (5, 0.75), (9, 1.5), (19, 3.5)]:
        ref = cv2.GaussianBlur(img, (ksz, ksz), sigma)
        assert np.abs(fb.gaussian_blur(img, ksz, sigma) - ref).max() < 2e-4
    for (w, h) in [(61, 38), (123, 77), (200, 150)]:
        ref = cv2.resize(img, (w, h), interpolation=cv2.INTER_LINEAR)
        assert np.abs(fb.resize_bilinear(img, w, h) - ref).max() < 2e-3   # white noise, 0..255 scale
