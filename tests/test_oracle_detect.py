"""CPU: FoE / phi / mask / metric restatements against vectors produced by the reference modules."""
import os

import numpy as np
import pytest

from oracle import ccl_np
from oracle import detect_np as dn


@pytest.mark.parametrize('ci', [0, 1, 2, 3])
def test_detect_oracle_reproduces_reference(golden_dir, ci):
    g = np.load(os.path.join(golden_dir, 'detect_%d.npz' % ci))
    fi = int(g['frame_index'])
    fd, foe, phi, total, fixed = dn.frame_pipeline(fi, g['flow'], g['ang'], float(g['dt']), g['sky'], g['ry'], g['rx'])
    assert fd.dtype == g['flow_derot'].dtype and np.array_equal(fd, g['flow_derot'])
    assert foe == (float(g['foe'][0]), float(g['foe'][1]))
    assert phi.dtype == g['phi'].dtype and np.array_equal(phi, g['phi'])
    assert np.array_equal(total, g['total_mask']) and np.array_equal(fixed, g['estimate_fixed'])
    assert dn.simple_bounding_box(g['seg']) == tuple(int(v) for v in g['bbox'])
    r = g['rates']
    assert dn.tpr_fpr(g['seg'], total) == (r[0], r[1])
    assert dn.tpr_fpr(g['seg'], fixed) == (r[2], r[3])


@pytest.mark.parametrize('ci', [0, 1, 2, 3])
def test_sample_indices_follow_the_legacy_rng(golden_dir, ci):
    g = np.load(os.path.join(golden_dir, 'detect_%d.npz' % ci))
    h, w = g['flow'].shape[:2]
    np.random.seed(int(g['seed']))
    ry, rx = dn.draw_sample_indices(h, w)
    assert np.array_equal(ry, g['ry']) and np.array_equal(rx, g['rx'])


def test_ransac_edge_cases():
    assert dn.ransac(np.zeros((0, 2))) == (0.0, 0.0)
    assert dn.ransac(np.array([[5.0, 5.0]])) == (0.0, 0.0)            # a lone estimate scores 0
    e = np.array([[0.0, 1.0], [100.0, 100.0], [101.0, 100.0], [1.0, 1.0]])
    assert dn.ransac(e) == (0.0, 1.0)                                  # first maximum wins ties


def test_bbox_and_rates_edge_cases():
    assert dn.simple_bounding_box(np.zeros((5, 7), np.uint8)) == (-1, -1, -1, -1)
    seg = np.zeros((5, 7), np.uint8)
    with np.errstate(all='ignore'):
        tpr, fpr = dn.tpr_fpr(seg, np.zeros((5, 7), bool))
    assert np.isnan(tpr) and fpr == 0.0


def test_ccl_oracles_agree():
    rng = np.random.default_rng(3)
    for shape, p in [((17, 23), 0.5), ((40, 64), 0.35), ((64, 40), 0.6), ((8, 8), 1.0), ((8, 8), 0.0)]:
        m = rng.random(shape) < p
        a = ccl_np.label_floodfill(m)
        b = ccl_np.label_scipy(m)
        assert np.array_equal(a, b)
        try:
            import cv2  # noqa: F401
            assert np.array_equal(a, ccl_np.label_cv2(m))
        except ImportError:
            pass
        lab, stats = ccl_np.label(m)
        assert stats.shape[0] == lab.max()
        if lab.max():
            assert stats[:, 4].sum() == m.sum()
        for i in range(lab.max()):
            ys, xs = np.nonzero(lab == i + 1)
            assert tuple(stats[i]) == (xs.min(), ys.min(), xs.max() - xs.min() + 1, ys.max() - ys.min() + 1, xs.size)
