"""GPU: Farneback over the whole parameter range mavd_create accepts and on frames down to 8 pixels a side.

Every accepted combination promises cv2.calcOpticalFlowFarneback's result.  Each case runs one pair through the CUDA
path and compares it level by level with the NumPy oracle (oracle/farneback_np.py, itself pinned against cv2 in
tests/test_oracle_farneback.py) and the final flow with live cv2, at the bars of test_gpu_farneback.py.  Each row of
the parameter table names the kernel branch it exists for."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPE_MEAN_TIGHT = 2e-5    # px, flow of every level against the oracle and final flow against cv2
EPE_MAX_TOL = 2e-3       # px, final flow against cv2
IMG_TOL = 5e-4           # pyramid image, 0..255 scale
REL_TOL = 2e-4           # R and M, relative to the largest magnitude of the plane set

KEYS = ('pyr_scale', 'levels', 'winsize', 'iterations', 'poly_n', 'poly_sigma', 'flags')


def _params(*p):
    return dict(zip(KEYS, p))


def _frames(w, h, seq=7):
    """One pair of w x h: synthetic frames when the generator can build them, else a crop of a 64 x 64 pair."""
    from mav_detection_b200 import synth
    if w >= 64 and h >= 64:
        return synth.make_pair(w, h, seq=seq)
    a, b = synth.make_pair(64, 64, seq=seq)
    y0, x0 = (64 - h) // 2, (64 - w) // 2
    return np.ascontiguousarray(a[y0:y0 + h, x0:x0 + w]), np.ascontiguousarray(b[y0:y0 + h, x0:x0 + w])


def _run(eng, prev, nxt):
    """Flow of one pair plus every tap: [(img0, img1, R0, R1, M, flow) per level], level 0's flow = the output."""
    import torch
    frames = torch.from_numpy(np.stack([prev, nxt])).cuda()
    flow = eng.farneback(frames, pair_stride=2)
    torch.cuda.synchronize()
    eng._keep_alive = (frames, flow)     # the level-0 taps read the caller's buffers of the last call
    flow = flow[0].cpu().numpy()
    levels = []
    for lvl in range(len(eng.levels)):
        t = [eng.tap('img', lvl, j).cpu().numpy() for j in (0, 1)] + [eng.tap('R', lvl, j).cpu().numpy() for j in (0, 1)]
        t.append(eng.tap('M', lvl, 0).cpu().numpy())
        t.append(flow if lvl == 0 else eng.tap('flow', lvl, 0).cpu().numpy())
        levels.append(t)
    return flow, levels


def _check_against_oracle_and_cv2(prev, nxt, p, flow, levels):
    cv2 = pytest.importorskip('cv2')
    from oracle import farneback_np as fb
    taps = {}
    fb.calc_optical_flow_farneback(prev, nxt, None, *[p[k] for k in KEYS],
                                   tap=lambda n, l, a: taps.__setitem__((n, l), a.copy()))
    h, w = prev.shape
    assert len(levels) == len(fb.level_schedule(w, h, p['pyr_scale'], p['levels']))
    last = p['iterations'] - 1
    for lvl, (i0, i1, R0, R1, M, fl) in enumerate(levels):
        for j, (img, R) in enumerate(((i0, R0), (i1, R1))):
            assert np.abs(img - taps[('img%d' % j, lvl)]).max() < IMG_TOL, ('img', lvl, j)
            ref = taps[('R%d' % j, lvl)]
            assert np.abs(R - ref).max() < REL_TOL * max(1.0, np.abs(ref).max()), ('R', lvl, j)
        # the matrices after the last UpdateMatrices of the level (M0 when there is a single iteration)
        ref = taps[('M%d' % last, lvl)]
        assert np.abs(M - ref).max() < REL_TOL * max(1.0, np.abs(ref).max()), ('M', lvl, float(np.abs(M - ref).max()))
        epe = np.linalg.norm(fl - taps[('flow%d' % last, lvl)], axis=-1).mean()
        assert epe < EPE_MEAN_TIGHT, ('flow', lvl, epe)
    ref = cv2.calcOpticalFlowFarneback(prev, nxt, None, *[p[k] for k in KEYS])
    epe = np.linalg.norm(flow - ref, axis=-1)
    assert epe.mean() < EPE_MEAN_TIGHT and epe.max() < EPE_MAX_TOL, ('cv2', epe.mean(), epe.max())
    assert np.linalg.norm(ref, axis=-1).max() > 0.01         # the pair moves: the comparison is not vacuous


def _staged_stride(src, dst):
    """Smallest distance between the first source samples of adjacent outputs of a resize src -> dst (api.cu:
    hstride_min); the staged horizontal pyramid pass runs on levels where it is >= 8."""
    from oracle import farneback_np as fb
    i0 = fb._resize_axis_coeffs(src, dst)[0]
    return int(np.diff(i0).min())


# (id, W, H, params, tuning) — the id names the branch the row exists for
TABLE = [
    # pyr_scale other than 0.5: levels that are not exact decimations (generic pyramid tables), the F64 resize
    # coordinates of matrices_init, and a coarsest level at stride >= 8 (staged horizontal pass)
    ('scale0.3-staged', 453, 371, _params(0.3, 5, 15, 3, 5, 1.2, 0), {}),
    ('scale0.65-staged', 453, 371, _params(0.65, 6, 15, 3, 5, 1.2, 0), {}),
    ('scale0.3-ragged', 333, 251, _params(0.3, 3, 13, 3, 5, 1.1, 0), {}),
    ('scale0.65-ragged', 333, 251, _params(0.65, 4, 15, 2, 7, 1.5, 256), {}),
    # 16 pyramid images: the whole PyrDesc and the level cap
    ('scale0.9-16-images', 320, 240, _params(0.9, 15, 15, 2, 5, 1.2, 0), {}),
    # generic iteration kernel at m = 11..31: column halo up to 32, ~105 KB of shared memory, windows wider than the
    # 50 x 36 coarsest level
    ('win23-box', 200, 144, _params(0.5, 3, 23, 3, 5, 1.2, 0), {}),
    ('win23-gauss', 200, 144, _params(0.5, 3, 23, 3, 5, 1.2, 256), {}),
    ('win33-box', 200, 144, _params(0.5, 3, 33, 3, 5, 1.2, 0), {}),
    ('win33-gauss', 200, 144, _params(0.5, 3, 33, 3, 5, 1.2, 256), {}),
    ('win47-box', 200, 144, _params(0.5, 3, 47, 2, 5, 1.2, 0), {}),
    ('win47-gauss', 200, 144, _params(0.5, 3, 47, 2, 7, 1.5, 256), {}),
    ('win63-box', 200, 144, _params(0.5, 3, 63, 2, 5, 1.2, 0), {}),
    ('win63-gauss', 200, 144, _params(0.5, 3, 63, 2, 7, 1.5, 256), {}),
    # one iteration: the last (fused) iteration launched straight after matrices_init, on both tile heights of the
    # TMA kernel (m = 7) and on the generic kernel (m = 10)
    ('iter1-tma-small-tiles', 320, 240, _params(0.5, 3, 15, 1, 5, 1.2, 0), dict(iter_small_tiles=1)),
    ('iter1-tma-full-tiles', 320, 240, _params(0.5, 3, 15, 1, 5, 1.2, 0), dict(iter_small_tiles=0)),
    ('iter1-tma-gauss', 320, 240, _params(0.5, 3, 13, 1, 5, 1.2, 256), {}),
    ('iter1-generic', 320, 240, _params(0.5, 3, 21, 1, 5, 1.2, 0), {}),
    # PolyExp with n outside {3, 5, 7, 8} (PE_LAUNCH(0)) and the poly_sigma < eps branch (sigma = 0.3 n)
    ('poly1', 320, 240, _params(0.5, 3, 15, 3, 1, 1.1, 0), {}),
    ('poly2', 320, 240, _params(0.5, 3, 15, 3, 2, 1.1, 0), {}),
    ('poly4', 320, 240, _params(0.5, 3, 15, 3, 4, 1.2, 0), {}),
    ('poly6-sigma3', 320, 240, _params(0.5, 3, 15, 3, 6, 3.0, 0), {}),
    ('poly5-sigma0', 320, 240, _params(0.5, 3, 15, 3, 5, 0.0, 0), {}),
    ('poly8', 320, 240, _params(0.4, 2, 12, 4, 8, 1.8, 0), {}),
]


@pytest.mark.parametrize('name,w,h,p,tuning', TABLE, ids=[r[0] for r in TABLE])
def test_parameter_table_stage_by_stage(name, w, h, p, tuning):
    from mav_detection_b200 import engine
    prev, nxt = _frames(w, h)
    eng = engine.Engine(w, h, p, max_pairs=1)
    if tuning:
        eng.set_tuning(**tuning)
    if name.endswith('-staged'):
        cw, ch = eng.levels[-1]
        assert _staged_stride(w, cw) >= 8, eng.levels
    if name == 'scale0.9-16-images':
        assert len(eng.levels) == 16
    if p['winsize'] >= 47:
        assert min(eng.levels[-1]) < p['winsize'], eng.levels       # a window wider than the coarsest level
    flow, levels = _run(eng, prev, nxt)
    _check_against_oracle_and_cv2(prev, nxt, p, flow, levels)
    eng.close()


TINY_SIZES = [(8, 8), (9, 9), (8, 64), (64, 8), (9, 12), (10, 10), (16, 8), (16, 16), (24, 40), (31, 33), (32, 32),
              (48, 17)]
TINY_PARAMS = {
    'c2': _params(0.5, 5, 15, 3, 5, 1.2, 0),
    'reference': _params(0.4, 1, 12, 10, 8, 1.2, 0),
    'win21-gauss': _params(0.5, 3, 21, 3, 7, 1.5, 256),
    'win63-box': _params(0.5, 3, 63, 2, 5, 1.2, 0),
}


@pytest.mark.parametrize('pname', list(TINY_PARAMS))
@pytest.mark.parametrize('size', TINY_SIZES, ids=['%dx%d' % s for s in TINY_SIZES])
def test_tiny_frames(size, pname):
    """Single-level pyramids on frames smaller than the TMA boxes and tiles; sides of 8 and 9 pixels, where the border
    gate of UpdateMatrices wraps; widths that are multiples of 16 (level-0 expansion through TMA) and widths that are
    not."""
    from mav_detection_b200 import engine
    w, h = size
    p = TINY_PARAMS[pname]
    prev, nxt = _frames(w, h, seq=3)
    eng = engine.Engine(w, h, p, max_pairs=1)
    assert eng.levels == [(w, h)]
    flow, levels = _run(eng, prev, nxt)
    _check_against_oracle_and_cv2(prev, nxt, p, flow, levels)
    eng.close()


def _check_against_chained_oracle(seq, params, flow, fixed, rec, samples, first_index=0):
    """records / masks of every pair against the oracle chained on OUR flow (bit-exact stages), boxes against the
    labelling oracle, and the flow itself against cv2."""
    import cv2
    from oracle import ccl_np
    from oracle import detect_np as dn
    for p in range(flow.shape[0]):
        ref = cv2.calcOpticalFlowFarneback(seq.frames[p], seq.frames[p + 1], None, *[params[k] for k in KEYS])
        epe = np.linalg.norm(flow[p] - ref, axis=-1).mean()
        assert epe < 1e-3, (p, epe)
        fd, foe, phi, total, fix = dn.frame_pipeline(first_index + p, flow[p], seq.omega[p + 1], seq.dt, seq.sky_mask,
                                                     samples[p, :2000], samples[p, 2000:], cr_arccos_f32=True)
        assert tuple(rec[p]['foe']) == foe, (p, rec[p]['foe'], foe)
        assert np.array_equal(fixed[p].astype(bool), fix), (p, int((fixed[p].astype(bool) != fix).sum()))
        st = rec[p]['stats']
        assert st['n_total'] == total.sum() and st['n_fixed'] == fix.sum(), p
        seg = seq.segmentation[p + 1]
        assert st['positives'] == (seg > 127).sum() and st['negatives'] == ((255 - seg) > 127).sum()
        assert st['tp_total'] == (total & (seg > 127)).sum() and st['fp_total'] == (total & (seg <= 127)).sum()
        assert st['tp_fixed'] == (fix & (seg > 127)).sum() and st['fp_fixed'] == (fix & (seg <= 127)).sum()
        assert tuple(st['seg_bbox']) == dn.simple_bounding_box(seg)
        assert np.allclose(st['seg_flow_sum'], fd[seg > 127].astype(np.float64).sum(axis=0), rtol=1e-9)
        lab, stats = ccl_np.label(fixed[p])
        assert rec[p]['n_labels'] == lab.max(), p
        k = min(32, stats.shape[0])
        assert np.array_equal(rec[p]['boxes'][:k], stats[:k]), p


@pytest.mark.parametrize('size', [(8, 8), (9, 12), (31, 33), (48, 17)], ids=lambda s: '%dx%d' % s)
def test_whole_path_on_tiny_frames(size):
    """eng.process on crops of a rotating, translating 64 x 64 sequence: the second pair is derotated and the crop
    holds part of the segmented blob."""
    pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, synth
    from oracle import detect_np as dn
    w, h, n = size[0], size[1], 2
    full = synth.make_sequence(64, 64, n + 1, seq=9, with_rotation=True, motion='translate')
    y0, x0 = min(30, 64 - h), min(30, 64 - w)
    crop = (slice(None), slice(y0, y0 + h), slice(x0, x0 + w))
    seq = synth.SyntheticSequence(np.ascontiguousarray(full.frames[crop]), np.ascontiguousarray(full.segmentation[crop]),
                                  np.zeros((h, w), bool), full.foe, full.omega, full.dt)
    assert (seq.segmentation[1:] > 127).any()
    params = dict(engine.SAMPLE_PARAMS)
    np.random.seed(40 + w)
    samples = np.stack([np.concatenate(dn.draw_sample_indices(h, w)) for _ in range(n)]).astype(np.int32)
    eng = engine.Engine(w, h, params, max_pairs=n)
    imu = engine.make_imu(n, seq.omega[1:n + 1], seq.dt, derotate=[i >= 1 for i in range(n)])
    flow_t = torch.empty((n, h, w, 2), dtype=torch.float32, device=eng.device)
    fixed_t = torch.empty((n, h, w), dtype=torch.uint8, device=eng.device)
    rec = eng.process(torch.from_numpy(seq.frames).to(eng.device), imu, torch.from_numpy(samples).to(eng.device),
                      seg=torch.from_numpy(seq.segmentation[1:n + 1].copy()).to(eng.device), flow_out=flow_t,
                      fixed_out=fixed_t)
    _check_against_chained_oracle(seq, params, flow_t.cpu().numpy(), fixed_t.cpu().numpy(),
                                  eng.records_to_numpy(rec), samples)
    eng.close()


def _narrow_masks(w, h):
    """full, checkerboard, vertical stripes, diagonals (both directions), noise."""
    y, x = np.mgrid[0:h, 0:w]
    rng = np.random.default_rng(w)
    return np.stack([np.ones((h, w), bool), (x + y) % 2 == 0, x % 2 == 0, (x - y) % 3 == 0, (x + y) % 4 == 1,
                     rng.random((h, w)) < 0.45]).astype(np.uint8)


@pytest.mark.parametrize('w', [8, 9, 16, 31, 33])
def test_labelling_and_wire_format_at_narrow_widths(w):
    """Below 32 pixels a row, one 128-pixel unit of the run-based labelling spans more than 4 rows and a packed row
    is not a whole number of 32-bit words."""
    import torch
    from mav_detection_b200 import engine
    from oracle import ccl_np
    h = 37
    masks = _narrow_masks(w, h)
    masks[5] *= np.random.default_rng(1).integers(1, 256, (h, w)).astype(np.uint8)     # any non-zero byte is set
    n = masks.shape[0]
    eng = engine.Engine(w, h, engine.SAMPLE_PARAMS, max_pairs=n)
    dm = torch.from_numpy(masks).cuda()
    labels, boxes, cnt = eng.ccl(dm)
    labels, boxes, cnt = labels.cpu().numpy(), boxes.cpu().numpy(), cnt.cpu().numpy()
    for i in range(n):
        ref, stats = ccl_np.label(masks[i])
        assert cnt[i] == ref.max(), (i, cnt[i], ref.max())
        assert np.array_equal(labels[i], ref), i
        k = min(32, stats.shape[0])
        assert np.array_equal(boxes[i, :k], stats[:k]), i
        assert not boxes[i, k:].any(), i
    pb = eng.packed_mask_bytes
    bits = eng.pack_mask(dm).cpu().numpy()
    flat = np.packbits(masks.reshape(n, -1) != 0, axis=-1, bitorder='little')
    assert bits.shape == (n, pb) and pb * 8 >= w * h
    assert np.array_equal(bits[:, :flat.shape[1]], flat) and not bits[:, flat.shape[1]:].any()
    for value in (1, 255):
        back = eng.unpack_mask(torch.from_numpy(bits).cuda(), value).cpu().numpy()
        assert np.array_equal(back, (masks != 0).astype(np.uint8) * value), value
    eng.close()


@pytest.mark.parametrize('w,h,overrides', [
    (320, 240, dict(pyr_scale=0.9, levels=16)),      # 17 pyramid images
    (320, 240, dict(winsize=64)),
    (320, 240, dict(poly_n=9)),
    (7, 32, {}),
    (32, 7, {}),
], ids=['17-images', 'winsize64', 'poly_n9', 'width7', 'height7'])
def test_outside_the_accepted_range_raises(w, h, overrides):
    """cv2 accepts some of these; the CUDA path has no kernel for them and says so."""
    from mav_detection_b200 import engine
    p = dict(engine.SAMPLE_PARAMS)
    p.update(overrides)
    with pytest.raises(ValueError):
        engine.Engine(w, h, p, max_pairs=1)


def test_edges_of_the_accepted_range_build():
    """The last accepted value next to each rejected one; the parameter table and the tiny-frame cases compare their
    results with the oracle and cv2."""
    from mav_detection_b200 import engine
    for w, h, overrides, n_levels in [(320, 240, dict(pyr_scale=0.9, levels=15), 16), (320, 240, dict(winsize=63), 3),
                                      (320, 240, dict(poly_n=8), 3), (8, 32, {}, 1), (32, 8, {}, 1)]:
        p = dict(engine.SAMPLE_PARAMS)
        p.update(overrides)
        eng = engine.Engine(w, h, p, max_pairs=1)
        assert len(eng.levels) == n_levels, (overrides, eng.levels)
        eng.close()


def _taps_under(eng, prev, nxt, **tuning):
    eng.set_tuning(**tuning)
    flow, levels = _run(eng, prev, nxt)
    return [flow] + [a for lv in levels for a in lv]


@pytest.mark.parametrize('knob,values,p', [
    ('mat_coord', (1, 2), _params(0.3, 5, 15, 3, 5, 1.2, 0)),
    ('mat_coord', (1, 2), _params(0.8, 5, 15, 3, 5, 1.2, 0)),
    ('pyr_staged', (0,), _params(0.3, 5, 15, 3, 5, 1.2, 0)),
    ('iter_small_tiles', (0,), _params(0.3, 5, 15, 1, 5, 1.2, 0)),
    ('iter_small_tiles', (0,), _params(0.5, 3, 15, 1, 5, 1.2, 0)),
], ids=['mat_coord-0.3', 'mat_coord-0.8', 'pyr_staged-0.3', 'iter_small_tiles-iter1-0.3', 'iter_small_tiles-iter1'])
def test_kernel_selection_knobs_are_bit_identical(knob, values, p):
    """Launch-shape and data-path knobs at the scales where they select different code.  mat_coord 0 recomputes the
    resize coordinates in double (farneback.cu: resize_coord), 1 reads the host-built tables, 2 forbids the float32
    power-of-two form: the coordinates, and so every tap and the flow, must be the same bits."""
    from mav_detection_b200 import engine
    w, h = 453, 371
    prev, nxt = _frames(w, h, seq=5)
    eng = engine.Engine(w, h, p, max_pairs=1)
    default = eng.get_tuning()[knob]
    assert default not in values
    ref = _taps_under(eng, prev, nxt)
    for v in values:
        got = _taps_under(eng, prev, nxt, **{knob: v})
        for i, (a, b) in enumerate(zip(got, ref)):
            assert np.array_equal(a, b), (knob, v, i, float(np.abs(a - b).max()))
    eng.set_tuning(**{knob: default})
    eng.close()
