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


DEFAULTS = dict(magnitude_threshold=2.5, ransac_threshold=30.0, dyn_offset=0.25, dyn_base=0.5, dyn_gain=8.0,
                dyn_min_mag=0.5, fixed_min_mag=1.0, fixed_angle=15.0)


@pytest.mark.parametrize('ci', [0, 1, 2, 3])
def test_explicit_default_parameters_are_the_reference_constants(golden_dir, ci):
    g = np.load(os.path.join(golden_dir, 'detect_%d.npz' % ci))
    fi = int(g['frame_index'])
    args = (fi, g['flow'], g['ang'], float(g['dt']), g['sky'], g['ry'], g['rx'])
    implicit = dn.frame_pipeline(*args)
    explicit = dn.frame_pipeline(*args, **DEFAULTS)
    assert implicit[1] == explicit[1]
    for a, b in zip(implicit[:1] + implicit[2:], explicit[:1] + explicit[2:]):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    fd = implicit[0]
    E = dn.intersections(fd, g['ry'], g['rx'], magnitude_threshold=2.5)
    assert np.array_equal(E, dn.intersections(fd, g['ry'], g['rx'])) and dn.ransac(E, 30.0) == dn.ransac(E)


def test_float32_frame_parameters_are_applied_in_float32():
    """NEP 50: Python-float parameters on the float32 frame act as their float32 values (what the CUDA path does)."""
    F = np.float32
    rng = np.random.default_rng(1)
    f = rng.normal(0, 2, (40, 50, 2)).astype(np.float32)
    foe = (20.3, 30.0)
    # magnitudes exactly at the float32 value of a gate, pointing at the FoE (phi = 180): float32(0.3) and float32(1.1)
    # lie above 0.3 and 1.1, so a float64 evaluation would let these pixels through both gates
    for x, m in ((40, F(0.3)), (41, F(1.1))):
        f[30, x] = (-m, 0.0)
    phi = dn.get_phi(f, foe, cr_arccos_f32=True)
    assert phi[30, 40] == phi[30, 41] == F(180)
    sky = np.zeros((40, 50), bool)
    sky[:3] = True
    p = dict(dyn_offset=0.1, dyn_base=0.3, dyn_gain=7.7, dyn_min_mag=0.3, fixed_min_mag=1.1, fixed_angle=14.9)
    total, fixed = dn.masks(f, phi, sky, **p)
    mag = np.linalg.norm(f, axis=-1)
    assert mag.dtype == np.float32 and phi.dtype == np.float32
    with np.errstate(divide='ignore'):
        t = F(0.3) + F(7.7) / mag
    assert t.dtype == np.float32
    amax, amin = phi > (F(0.1) + t), phi < (F(0.1) - t)
    ref_total = (mag > F(0.3)) & ~sky & (amin | amax)
    ref_fixed = np.where((mag > F(1.1)) & ~sky, phi, F(0)) > F(14.9)
    assert np.array_equal(total, ref_total) and np.array_equal(fixed, ref_fixed)
    assert not total[30, 40] and total[30, 41] and not fixed[30, 41]
    # the same values in float64 decide those pixels the other way
    t64, f64 = dn.masks(f.astype(np.float64), phi.astype(np.float64), sky, **p)
    assert t64[30, 40] and f64[30, 41]


def test_float32_foe_gate_compares_in_float32():
    """get_magnitude(flow2) < magnitude_threshold in the flow's dtype: float32(0.7) < 0.7, yet a float32 magnitude of
    float32(0.7) passes the float32 gate."""
    f = np.zeros((2, 3, 2), np.float32)
    f[0, 2] = (0.0, 1.0)                    # first points: the vertical line x = 2
    f[1, 0] = (np.float32(0.7), 0.0)        # second points: the horizontal line y = 1, |f| == float32(0.7)
    ry = np.r_[np.zeros(1000, int), np.ones(1000, int)]
    rx = np.r_[np.full(1000, 2), np.zeros(1000, int)]
    E32 = dn.intersections(f, ry, rx, magnitude_threshold=0.7)
    assert E32.shape == (1000, 2) and (E32 == (2.0, 1.0)).all()
    assert dn.intersections(f.astype(np.float64), ry, rx, magnitude_threshold=0.7).shape[0] == 0
    assert dn.foe_dense(f, ry, rx, magnitude_threshold=0.7) == (2.0, 1.0)


def _direct_counts(gt, mask):
    g = gt.astype(np.int64)
    m = mask.astype(bool)
    return (int((g > 127).sum()), int((g <= 127).sum()), int(((g >= 1) & m).sum()), int(((g <= 254) & m).sum()))


@pytest.mark.parametrize('mx', [255, 100, 30, 10, 1, 0])
def test_graded_segmentation_metrics_match_direct_counts(mx):
    """tpr_fpr and simple_bounding_box on graded uint8 masks: g > 127 positives, g >= 1 true and g <= 254 false
    positives of a 0/1 mask, box of g > 0.1 * max."""
    rng = np.random.default_rng(mx)
    h, w = 23, 31
    special = np.array([0, 1, 126, 127, 128, 254, 255])
    seg = rng.choice(special[special <= mx], (h, w)).astype(np.uint8)
    seg[rng.random((h, w)) < 0.3] = 0
    if mx:
        seg = np.minimum(seg, mx).astype(np.uint8)
        seg[rng.integers(h), rng.integers(w)] = mx
    mask = rng.random((h, w)) < 0.5
    assert dn.metric_counts(seg, mask) == _direct_counts(seg, mask)
    p, n, tp, fp = _direct_counts(seg, mask)
    with np.errstate(divide='ignore', invalid='ignore'):
        assert dn.tpr_fpr(seg, mask) == (np.float64(tp) / p, np.float64(fp) / n) or p == 0
    if p == 0:
        tpr, fpr = dn.tpr_fpr(seg, mask)
        assert (np.isnan(tpr) if tp == 0 else np.isinf(tpr)) and fpr == fp / n
    # box: integer threshold floor(0.1 * max) + 1 (0.1 * 10 == 1.0 exactly, 0.1 * 30 == 3.0000000000000004)
    smin = int(np.floor(0.1 * int(seg.max()))) + 1
    ys, xs = np.nonzero(seg.astype(np.int64) >= smin)
    ref = (-1, -1, -1, -1) if ys.size == 0 else (int(xs.min()), int(ys.min()), int(xs.max()), int(ys.max()))
    assert dn.simple_bounding_box(seg) == ref
    if mx in (10, 100):
        s2 = np.zeros((h, w), np.uint8)
        s2[5, 5] = mx
        s2[0, 30] = mx // 10                # exactly 0.1 * max: outside the box
        s2[22, 0] = mx // 10 + 1
        assert dn.simple_bounding_box(s2) == (0, 5, 5, 22)
