"""GPU: the sparse feature path (mavd_good_features_to_track, mavd_pyr_lk) against cv2 and oracle/lk_np.py.

Eig images are cv2.cornerMinEigenVal's bits, corner lists cv2.goodFeaturesToTrack's, tracker status
cv2.calcOpticalFlowPyrLK's on every point, positions and err within the bars of tests/test_oracle_lk.py.  A pair's or a
frame's results do not depend on the batch that carries it."""
import cv2
import numpy as np
import pytest
import torch

from mav_detection_b200 import _lib, engine, lucas_kanade, synth
from oracle import lk_np as lk
from test_oracle_lk import LK_CASES, _lk_points, check_lk, frame_pair

pytestmark = pytest.mark.gpu
TC, TE = cv2.TERM_CRITERIA_COUNT, cv2.TERM_CRITERIA_EPS


def _eng(W, H, max_pairs=1):
    return engine.Engine(W, H, max_pairs=max_pairs)


def _corners(c, n, i):
    k = min(int(n[i]), c.shape[1])
    return c[i, :k].cpu().numpy()


@pytest.mark.parametrize('W,H', [(8, 8), (33, 17), (640, 480), (1920, 1080), (3840, 2160)])
def test_eig_and_corners_match_cv2(W, H):
    a, b = frame_pair(W, H)
    eng = _eng(W, H, 1)
    fr = torch.from_numpy(np.stack([a, b])).cuda()
    for bs in ((1, 2, 3, 7, 31) if W < 3000 else (7,)):
        ref_eig = cv2.cornerMinEigenVal(a, bs, ksize=3)
        for q in (1e-4, 0.01, 0.3, 1.0):
            for md in ((0, 0.5, 1, 7, 7.4, 30) if W < 1000 else (7,)):
                c, n, eig = eng.good_features(fr, 2000, q, md, bs, want_eig=True)
                if q == 0.01 and md == 0:
                    e = eig[0].cpu().numpy()
                    assert np.array_equal(e.view(np.int32), ref_eig.view(np.int32)), (W, bs)
                    if W < 1000:
                        assert np.array_equal(e, lk.corner_min_eig_val(a, bs))
                for mc in (0, 1, 25, 2000):
                    ref = cv2.goodFeaturesToTrack(a, mc, q, md, blockSize=bs)
                    if mc == 0:
                        if ref is None:
                            assert int(n[0]) == 0
                            continue
                        assert int(n[0]) == len(ref), (bs, q, md)
                        cc, nn = eng.good_features(fr[:1], int(n[0]), q, md, bs)
                        assert np.array_equal(_corners(cc, nn, 0), ref.reshape(-1, 2)), (bs, q, md)
                    else:
                        got = _corners(c, n, 0)[:mc]
                        if ref is None:
                            assert len(got) == 0
                        else:
                            assert np.array_equal(got, ref.reshape(-1, 2)), (bs, q, md, mc)
    eng.close()


def test_corner_masks_and_constant_frame():
    W, H = 640, 480
    eng = _eng(W, H, 2)
    a, b = frame_pair(W, H)
    rng = np.random.default_rng(5)
    m0 = (rng.integers(0, 2, (H, W)) * 255).astype(np.uint8)
    m1 = np.zeros((H, W), np.uint8)
    m1[50:400, 100:500] = 1
    fr = torch.from_numpy(np.stack([a, b])).cuda()
    # shared mask
    c, n = eng.good_features(fr, 500, 0.01, 5, 3, mask=torch.from_numpy(m0).cuda())
    for i, img in enumerate((a, b)):
        ref = cv2.goodFeaturesToTrack(img, 500, 0.01, 5, mask=m0, blockSize=3).reshape(-1, 2)
        assert np.array_equal(_corners(c, n, i), ref)
    # per-frame masks
    c, n = eng.good_features(fr, 500, 0.01, 5, 3, mask=torch.from_numpy(np.stack([m0, m1])).cuda())
    for i, (img, m) in enumerate(((a, m0), (b, m1))):
        ref = cv2.goodFeaturesToTrack(img, 500, 0.01, 5, mask=m, blockSize=3).reshape(-1, 2)
        assert np.array_equal(_corners(c, n, i), ref)
    # an empty mask and a constant frame give no corner (cv2: None)
    c, n = eng.good_features(fr, 10, 0.01, 5, 3, mask=torch.zeros((H, W), dtype=torch.uint8, device='cuda'))
    assert n.tolist() == [0, 0] and not c.any()
    z = torch.full((1, H, W), 77, dtype=torch.uint8, device='cuda')
    assert int(eng.good_features(z, 10, 0.01, 3)[1][0]) == 0
    assert lucas_kanade.goodFeaturesToTrack(np.full((H, W), 77, np.uint8), 10, 0.01, 3) is None
    eng.close()


@pytest.mark.parametrize('W,H', [(8, 8), (80, 60), (640, 480), (1920, 1080)])
def test_lk_matches_cv2_and_oracle(W, H):
    a, b = frame_pair(W, H)
    eng = _eng(W, H, 1)
    fr = torch.from_numpy(np.stack([a, b])).cuda()
    q = _lk_points(a, W, H, np.random.default_rng(W))
    q = np.concatenate([q, np.array([[np.nan, 1], [2, np.inf], [-np.inf, np.nan]], np.float32)])
    extra = [((21, 21), ml, 0, (TC | TE, 30, 0.01), me) for ml in range(9) for me in (0, 1e-4, 1e-2)]
    for win, ml, fl, cr, me in LK_CASES + extra:
        nx, st, er = eng.pyr_lk(fr, torch.from_numpy(q).cuda()[None], pair_stride=2, win=win, max_level=ml,
                                criteria=cr, flags=fl, min_eig_threshold=me)
        got = (nx[0].cpu().numpy(), st[0].cpu().numpy(), er[0].cpu().numpy())
        ref = cv2.calcOpticalFlowPyrLK(a, b, q[:-3].reshape(-1, 1, 2), None, winSize=win, maxLevel=ml, criteria=cr,
                                       flags=fl, minEigThreshold=me)
        check_lk(ref, (got[0][:-3], got[1][:-3], got[2][:-3]), win)
        assert got[1][-3:].tolist() == [0, 0, 0] and got[2][-3:].tolist() == [0, 0, 0]
        orc = lk.calc_optical_flow_pyr_lk(a, b, q, win, ml, cr, fl, me)
        assert np.array_equal(got[1], orc[1])
        ok = got[1] == 1
        assert np.array_equal(got[0][ok], orc[0][ok]), (win, ml, fl, cr, me)
        assert np.array_equal(got[2][ok], orc[2][ok])
    eng.close()


def test_batches_are_invariant_and_feed_each_other():
    W, H = 640, 480
    seq = synth.make_sequence(W, H, 66, seq=1, with_rotation=True)
    frames = torch.from_numpy(np.ascontiguousarray(seq.frames)).cuda()
    eng = _eng(W, H, 64)
    c, n = eng.good_features(frames[:65], 400, 0.01, 7, 7)
    for i in (0, 17, 64):
        ref = cv2.goodFeaturesToTrack(seq.frames[i], 400, 0.01, 7, blockSize=7).reshape(-1, 2)
        assert np.array_equal(_corners(c, n, i), ref)
    c1, n1 = eng.good_features(frames[17:18], 400, 0.01, 7, 7)
    assert torch.equal(c1[0], c[17]) and int(n1[0]) == int(n[17])
    full = eng.pyr_lk(frames, c[:64], n_points=n[:64], pair_stride=1)
    for p in (0, 31, 63):
        k = min(int(n[p]), 400)
        ref = cv2.calcOpticalFlowPyrLK(seq.frames[p], seq.frames[p + 1], c[p, :k].cpu().numpy().reshape(-1, 1, 2), None)
        check_lk(ref, tuple(t[p, :k].cpu().numpy() for t in full), (21, 21))
        assert not full[1][p, k:].any()
    for nb in (1, 5, 13):
        for start in (0, 3):
            sub = eng.pyr_lk(frames[start:start + nb + 1], c[start:start + nb].contiguous(),
                             n_points=n[start:start + nb].contiguous(), pair_stride=1)
            for t, u in zip(sub, full):
                assert torch.equal(t, u[start:start + nb])
    # stride 2 on the same pairs
    pairs = torch.stack([frames[:13], frames[1:14]], 1).reshape(26, H, W).contiguous()
    s2 = eng.pyr_lk(pairs, c[:13].contiguous(), n_points=n[:13].contiguous(), pair_stride=2)
    for t, u in zip(s2, full):
        assert torch.equal(t, u[:13])
    eng.close()


def test_rejections_allocate_nothing():
    W, H = 64, 48
    eng = _eng(W, H, 2)
    base = eng.workspace_bytes
    fr = torch.zeros((4, H, W), dtype=torch.uint8, device='cuda')
    pts = torch.zeros((2, 5, 2), dtype=torch.float32, device='cuda')
    for kw in (dict(block_size=0), dict(block_size=32), dict(quality_level=0.0), dict(min_distance=-1.0),
               dict(quality_level=float('nan')), dict(min_distance=float('nan')), dict(max_corners=-1)):
        args = dict(max_corners=10, quality_level=0.01, min_distance=3.0, block_size=3)
        args.update(kw)
        with pytest.raises(ValueError):
            eng.good_features(fr, **args) if args['max_corners'] >= 0 else \
                _lib.check(eng.lib.mavd_good_features_to_track(eng._h, fr.data_ptr(), 1, _lib.GfttParams(-1, 0.01, 3, 3, 3),
                                                                None, 0, None, pts.data_ptr(), None, None))
    with pytest.raises(ValueError):
        _lib.check(eng.lib.mavd_good_features_to_track(eng._h, fr.data_ptr(), 5, _lib.GfttParams(1, 0.01, 3, 3, 3),
                                                        None, 0, pts.data_ptr(), pts.data_ptr(), None, None))
    with pytest.raises(ValueError):
        _lib.check(eng.lib.mavd_good_features_to_track(eng._h, fr.data_ptr(), 1, _lib.GfttParams(1, 0.01, 3, 3, 5),
                                                        None, 0, pts.data_ptr(), pts.data_ptr(), None, None))
    for kw in (dict(win=(2, 21)), dict(win=(21, 64)), dict(max_level=-1), dict(max_level=_lib.LK_MAX_LEVEL + 1),
               dict(flags=4), dict(flags=1), dict(criteria=(TC, 10, float('nan'))), dict(min_eig_threshold=float('nan')),
               dict(criteria=(4, 10, 0.1)), dict(pair_stride=3)):
        with pytest.raises(ValueError):
            eng.pyr_lk(fr, pts, **kw)
    with pytest.raises(ValueError):
        _lib.check(eng.lib.mavd_pyr_lk(eng._h, fr.data_ptr(), 3, 1, _lib.LkParams(21, 21, 3, 3, 30, 0.01, 0, 1e-4),
                                       pts.data_ptr(), 5, None, pts.data_ptr(), pts.data_ptr(), pts.data_ptr(), None))
    with pytest.raises(ValueError):
        _lib.check(eng.lib.mavd_pyr_lk(eng._h, fr.data_ptr(), 1, 1, _lib.LkParams(21, 21, 3, 3, 30, 0.01, 0, 1e-4),
                                       None, 5, None, pts.data_ptr(), pts.data_ptr(), pts.data_ptr(), None))
    assert eng.workspace_bytes == base
    eng.good_features(fr, 5, 0.01, 3)
    assert eng.workspace_bytes > base
    quiet = _eng(W, H, 2)
    assert quiet.workspace_bytes == base
    quiet.close()
    eng.close()


def test_module_functions_return_what_cv2_returns():
    a, b = frame_pair(320, 240)
    for mc, q, md, bs in ((100, 0.01, 7, 3), (0, 0.05, 5, 7), (3, 0.3, 0, 2)):
        ref = cv2.goodFeaturesToTrack(a, mc, q, md, blockSize=bs)
        got = lucas_kanade.goodFeaturesToTrack(a, mc, q, md, blockSize=bs)
        assert got.dtype == ref.dtype and got.shape == ref.shape and np.array_equal(got, ref)
    p = cv2.goodFeaturesToTrack(a, 200, 0.01, 7)
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None)
    got = lucas_kanade.calcOpticalFlowPyrLK(a, b, p, None)
    for r, g in zip(ref, got):
        assert r.dtype == g.dtype and r.shape == g.shape
    check_lk(ref, got, (21, 21))
    ref = cv2.calcOpticalFlowPyrLK(a, b, p, None, winSize=(15, 15), maxLevel=2, flags=cv2.OPTFLOW_LK_GET_MIN_EIGENVALS)
    got = lucas_kanade.calcOpticalFlowPyrLK(a, b, p, None, winSize=(15, 15), maxLevel=2,
                                            flags=cv2.OPTFLOW_LK_GET_MIN_EIGENVALS)
    check_lk(ref, got, (15, 15))
