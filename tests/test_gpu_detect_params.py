"""GPU: the detection stages over the whole range of mavd_detect_params and on graded segmentation masks.

Every other GPU test runs with mavd_default_detect_params and 0/255 segmentation masks, which leave several branches of
detect.cu unreached: the window in which the float32 pre-decision (FAST) of the residual stage may run, the guards of
pixel_fast, the exact path with `amin` live, sqrt_threshold for thresholds whose square is not the boundary, the float32
FoE magnitude gate, the graded-mask statistics of residual_kernel and seg_max_kernel, and graph replay after a parameter
change.  Each row of the tables below names the branch it exists for.  Bars as in test_gpu_detect.py: masks, counts,
boxes, labels and FoE bit-exact against the oracle (oracle/detect_np.py with the same parameters), flow sums to
rtol 1e-9, the float32 frame bit-exact against the oracle with a correctly rounded arccos."""
import math
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEFAULTS = dict(magnitude_threshold=2.5, ransac_threshold=30.0, dyn_offset=0.25, dyn_base=0.5, dyn_gain=8.0,
                dyn_min_mag=0.5, fixed_min_mag=1.0, fixed_angle=15.0)
MASK_KEYS = ('dyn_offset', 'dyn_base', 'dyn_gain', 'dyn_min_mag', 'fixed_min_mag', 'fixed_angle')
COUNT_KEYS = ('n_total', 'n_fixed', 'positives', 'negatives', 'tp_total', 'fp_total', 'tp_fixed', 'fp_fixed')
NAN, INF = float('nan'), float('inf')


def _engine(w, h, n=1):
    from mav_detection_b200 import engine
    return engine.Engine(w, h, engine.SAMPLE_PARAMS, max_pairs=n)


def _full(p):
    d = dict(DEFAULTS)
    d.update({k: float(v) for k, v in p.items()})
    return d


def _set_params(eng, p):
    for k, v in _full(p).items():
        setattr(eng.detect_params, k, v)


def _mask_params(p):
    """The mask keywords of the oracle, as Python floats (NEP 50: they act in the frame's own precision)."""
    return {k: float(p[k]) for k in MASK_KEYS}


def _fast_enabled(p):
    """detect.cu residual_run: the parameter window in which the float32 pre-decision may run (phi not requested)."""
    return (p['fixed_angle'] >= 0.0 and p['dyn_gain'] >= 0.0 and p['dyn_offset'] - p['dyn_base'] < -1e-2 and
            p['dyn_min_mag'] >= 0.0 and p['fixed_min_mag'] >= 0.0 and p['fixed_angle'] <= 170.0 and
            p['dyn_offset'] + p['dyn_base'] < 160.0 and p['dyn_gain'] < 1e6 and p['dyn_min_mag'] < 1e3 and
            p['fixed_min_mag'] < 1e3)


def _sums_close(got, vals):
    """A float64 atomic sum against NumPy's: rtol 1e-9, and an absolute slack of 1e-9 of the summed magnitudes for
    sums that cancel."""
    vals = np.asarray(vals, np.float64).reshape(-1, 2)
    return np.allclose(got, vals.sum(axis=0), rtol=1e-9, atol=1e-9 * float(np.abs(vals).sum()) + 1e-300)


# ------------------------------------------------------------------------------------------------
# A. Residual stage over the parameter range
# ------------------------------------------------------------------------------------------------
W, H = 128, 48
FOE = (61.0, 15.0)          # on a pixel (phi at the FoE itself), and row 15 is exactly radial (phi = 0 / 180)

# (row id, parameters other than the defaults, branch)
ROWS = [
    ('defaults', {}, 'control'),
    ('fixed0', dict(fixed_angle=0.0), 'sf = crs: phi = 0 and 180 fall inside the guard'),
    ('fixed90', dict(fixed_angle=90.0), 'cos T = 0'),
    ('fixed170', dict(fixed_angle=170.0), 'last fixed angle FAST accepts'),
    ('fixed170.5', dict(fixed_angle=170.5), 'exact path, max_phi reported'),
    ('fixed180', dict(fixed_angle=180.0), 'nothing passes the fixed test'),
    ('fixed-1', dict(fixed_angle=-1.0), 'every pixel passes (0 > -1), sky and still pixels included; FAST off'),
    ('offset0.4899999', dict(dyn_offset=0.4899999), 'offset - base < -0.01: FAST'),
    ('offset0.4900001', dict(dyn_offset=0.4900001), 'offset - base >= -0.01: exact path'),
    ('offset20', dict(dyn_offset=20.0), 'amin live, exact path'),
    ('gain0', dict(dyn_gain=0.0), 'constant dynamic threshold'),
    ('gain100', dict(dyn_gain=100.0), 'threshold >= 170 and >= 180 deg for |f| in (0.5, 0.59): pixel_fast thr < 170'),
    ('gain999999', dict(dyn_gain=999999.0), 'last gain FAST accepts'),
    ('gain1e6', dict(dyn_gain=1e6), 'exact path'),
    ('minmag0', dict(dyn_min_mag=0.0, fixed_min_mag=0.0), 'gates at zero: zero and denormal flows'),
    ('minmag999.9', dict(dyn_min_mag=999.9, fixed_min_mag=999.9), 'last magnitude gates FAST accepts'),
    ('minmag1000', dict(dyn_min_mag=1000.0, fixed_min_mag=1000.0), 'magnitude gates outside FAST'),
    ('c0_159.9', dict(dyn_offset=79.45, dyn_base=80.45), 'offset + base < 160: FAST, thresholds up to 176 deg'),
    ('c0_160', dict(dyn_offset=79.5, dyn_base=80.5), 'offset + base = 160: exact path'),
    ('nonrepr', dict(dyn_offset=0.1, dyn_base=0.3, dyn_gain=7.7, dyn_min_mag=0.3, fixed_min_mag=1.1, fixed_angle=14.9),
     'values float32 rounds: the float32 frame applies them in float32'),
] + [('nan_' + k, {k: NAN}, 'NaN: exact path, NumPy comparison semantics') for k in MASK_KEYS] + [
    ('gain_inf', dict(dyn_gain=INF), 'infinite gain: exact path'),
]

MODES = ('rot', 'norot', 'f32')   # derotating with a rotation, derotating with a zero rotation (48-register build), float32
ANG_ROT, DT = np.array([0.002, -0.001, 0.0005]), 1 / 30


def _adversarial_field(h, w, foe, rng, p):
    """Flow (float64, in the derotated frame) whose angle to the FoE ray sits within 1e-9 .. 1e-1 degrees of the fixed
    threshold, of offset + base + gain/|f| and of offset - base - gain/|f| (where positive), with magnitudes hugging
    both gates (some exactly at the gate's float32 value), exactly radial flow, the FoE pixel, zero, denormal, NaN and
    inf flows, and small flows at small phi (where the sine test of pixel_fast breaks once the threshold reaches 180)."""
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    theta = np.arctan2(ys - foe[1], xs - foe[0])
    gates = [g for g in (p['dyn_min_mag'], p['fixed_min_mag']) if math.isfinite(g) and g > 0]
    s = max([1.0] + [g / 6.0 for g in gates])
    mag = rng.uniform(0.3 * s, 12.0 * s, (h, w))
    pick = rng.random((h, w))
    for i, g in enumerate(gates):
        near = (pick >= 0.1 * i) & (pick < 0.1 * i + 0.1)
        mag = np.where(near, g * (1.0 + rng.choice([-1, 1], (h, w)) * 10.0 ** rng.uniform(-9, -4, (h, w))), mag)
    small = (pick >= 0.2) & (pick < 0.3)
    mag = np.where(small, rng.uniform(0.5, 0.59, (h, w)), mag)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = p['dyn_base'] + p['dyn_gain'] / mag
        cands = np.stack([np.full((h, w), p['fixed_angle']), p['dyn_offset'] + t, p['dyn_offset'] - t])
    ok = np.isfinite(cands) & (cands >= 0.0) & (cands <= 180.0)
    which = rng.integers(0, 3, (h, w))
    thr = np.take_along_axis(cands, which[None], 0)[0]
    thr = np.where(np.take_along_axis(ok, which[None], 0)[0], thr, rng.uniform(0.0, 180.0, (h, w)))
    thr = np.where(small, rng.uniform(0.0, 3.0, (h, w)), thr)
    eps = rng.choice([-1, 1], (h, w)) * 10.0 ** rng.uniform(-9, -1, (h, w))
    ang = theta + rng.choice([-1, 1], (h, w)) * np.deg2rad(np.clip(thr + eps, 0.0, 180.0))
    f = np.stack([mag * np.cos(ang), mag * np.sin(ang)], -1)
    fy, fx = int(foe[1]), int(foe[0])
    f[fy, :fx] = np.stack([rng.choice([-1, 1], fx) * rng.uniform(0.3, 12.0, fx) * s, np.zeros(fx)], -1)    # radial
    f[fy, fx + 1:] = np.stack([rng.choice([-1, 1], w - fx - 1) * rng.uniform(0.3, 12.0, w - fx - 1) * s,
                               np.zeros(w - fx - 1)], -1)
    f[fy, fx] = (3.0 * s, 1.0)                                  # the FoE pixel: |d| = 0
    # magnitudes exactly at the float32 value of each gate, one float32 step either side, along both axes
    row = h - 1
    x = 0
    for g in gates:
        g32 = np.float32(g)
        for v in (np.nextafter(g32, np.float32(0)), g32, np.nextafter(g32, np.float32(np.inf))):
            for vec in ((v, 0.0), (-v, 0.0), (0.0, v), (0.0, -v)):
                f[row, x] = vec
                x += 1
    for vec in ((0.0, 0.0), (1e-40, 0.0), (0.0, -1e-42), (1e-40, 1e-40), (np.nan, 1.0), (1.0, np.nan), (np.inf, 1.0),
                (-np.inf, 0.0), (np.nan, np.nan), (3e-39, 2e-39)):
        f[row, x] = vec
        x += 1
    f[row - 1, :16] = 0.0                                        # still pixels
    return f


def _graded_seg(h, w, rng):
    seg = np.zeros((h, w), np.uint8)
    seg[20:34, 70:110] = rng.choice([0, 1, 126, 127, 128, 254, 255], (14, 40))
    seg[22:30, 75:100] |= rng.integers(0, 256, (8, 25), dtype=np.uint8)
    return seg


def _offset_copy(t, offset):
    """A CUDA copy of t that starts `offset` bytes into a larger buffer: a misaligned view (forces VEC == 1)."""
    import torch
    nb = t.numel() * t.element_size()
    buf = torch.zeros(nb + offset, dtype=torch.uint8, device='cuda')
    view = buf[offset:offset + nb].view(t.dtype).reshape(t.shape)
    view.copy_(t)
    return view


@pytest.fixture(scope='module')
def eng_a():
    e = _engine(W, H)
    yield e
    e.close()


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('row', ROWS, ids=[r[0] for r in ROWS])
def test_residual_over_parameter_range(eng_a, row, mode):
    import torch
    from mav_detection_b200 import engine
    from oracle import detect_np as dn
    name, prm, branch = row
    p = _full(prm)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    want = _adversarial_field(H, W, FOE, rng, p)
    ang = ANG_ROT if mode == 'rot' else np.zeros(3)
    rot = dn.derotation_field(W, H, ang, DT) if mode == 'rot' else 0.0
    with np.errstate(invalid='ignore'):
        flow = (want + rot).astype(np.float32)
    sky = np.zeros((H, W), np.uint8)
    sky[:4, :40] = 1
    sky[4:6, :40] = 255
    seg = _graded_seg(H, W, rng)
    derot = mode != 'f32'
    with np.errstate(invalid='ignore', over='ignore'):
        fd = dn.derotate(1 if derot else 0, flow, ang, DT)
        phi = dn.get_phi(fd, FOE, cr_arccos_f32=True)
        total_ref, fixed_ref = dn.masks(fd, phi, sky != 0, **_mask_params(p))
    fast = derot and _fast_enabled(p)
    _set_params(eng_a, prm)
    imu = engine.make_imu(1, ang[None], DT, derotate=derot)
    foe_t = torch.tensor([FOE], dtype=torch.float64, device='cuda')
    base = dict(flow=torch.from_numpy(flow[None]).cuda(), sky=torch.from_numpy(sky).cuda(),
                seg=torch.from_numpy(seg).cuda())
    runs = {}
    for aligned in (True, False):
        t = base if aligned else dict(flow=_offset_copy(base['flow'], 8), sky=_offset_copy(base['sky'], 1),
                                      seg=_offset_copy(base['seg'], 1))
        if not aligned:
            assert t['flow'].data_ptr() % 16 == 8 and t['seg'].data_ptr() % 4 == 1
        for exact in (False, True):
            eng_a.force_exact_residual(exact)
            _, tot, fix, st = eng_a.residual_masks(t['flow'], imu, foe_t, sky=t['sky'], seg=t['seg'], want_phi=False)
            runs[(aligned, exact)] = (tot[0].cpu().numpy().astype(bool), fix[0].cpu().numpy().astype(bool),
                                      eng_a.stats_to_numpy(st)[0])
        eng_a.force_exact_residual(False)
    counts_t, counts_f = dn.metric_counts(seg, total_ref), dn.metric_counts(seg, fixed_ref)
    ref_counts = dict(n_total=total_ref.sum(), n_fixed=fixed_ref.sum(), positives=counts_t[0], negatives=counts_t[1],
                      tp_total=counts_t[2], fp_total=counts_t[3], tp_fixed=counts_f[2], fp_fixed=counts_f[3])
    for (aligned, exact), (tot, fix, st) in runs.items():
        where = (name, mode, 'aligned' if aligned else 'offset', 'exact' if exact else 'fast')
        assert np.array_equal(tot, total_ref), where + ('total', int((tot != total_ref).sum()))
        assert np.array_equal(fix, fixed_ref), where + ('fixed', int((fix != fixed_ref).sum()))
        for k in COUNT_KEYS:
            assert st[k] == ref_counts[k], where + (k,)
        assert tuple(st['seg_bbox']) == dn.simple_bounding_box(seg), where
        assert _sums_close(st['seg_flow_sum'], fd[seg > 127]), where
        if fast and not exact:
            assert st['max_phi'] == -1.0, where
        elif derot:
            assert abs(st['max_phi'] - float(phi.max())) < 1e-9, where + (st['max_phi'], float(phi.max()))
        else:
            assert st['max_phi'] == float(phi.max()), where
    # the row is not vacuous: both masks have both classes somewhere, or the row pins an all / nothing outcome
    if name not in ('fixed180', 'fixed-1', 'minmag1000', 'nan_dyn_min_mag', 'nan_fixed_min_mag', 'nan_fixed_angle',
                    'nan_dyn_offset', 'nan_dyn_base', 'nan_dyn_gain', 'gain_inf'):
        assert 0 < fixed_ref.sum() < fixed_ref.size, (name, mode)
    if name == 'fixed-1':
        assert fixed_ref.all()
    if name == 'fixed180':
        assert not fixed_ref.any()
    if name == 'offset20':
        with np.errstate(divide='ignore', invalid='ignore'):
            mag = np.linalg.norm(fd, axis=-1)
            amin = phi < (20.0 - (0.5 + 8.0 / mag))
        assert (amin & (mag > 0.5) & (sky == 0) & total_ref).any()      # pixels the amin branch alone marks


# ------------------------------------------------------------------------------------------------
# B. Graded segmentation and sky
# ------------------------------------------------------------------------------------------------
NB = 6
SEG_MAXIMA = (10, 255, 100, 30, 1, 0)     # frame 0 holds its maximum only in the tail of seg_max_kernel's 16-byte loop


def _graded_frames(w, h, rng):
    npx = w * h
    tail = npx % 16 or 16
    segs = np.zeros((NB, h, w), np.uint8)
    for f, mx in enumerate(SEG_MAXIMA):
        flat = segs[f].reshape(-1)
        if mx == 255:
            flat[:] = rng.integers(0, 256, npx)
            flat[rng.integers(0, npx, 40)] = rng.choice([0, 1, 126, 127, 128, 254, 255], 40)
        elif mx:
            # interior values below the maximum, with the values on either side of the box threshold 0.1 * max
            blob = np.zeros((h, w), np.uint8)
            blob[h // 3:2 * h // 3, w // 3:2 * w // 3] = rng.integers(0, mx, (2 * h // 3 - h // 3, 2 * w // 3 - w // 3))
            flat[:] = blob.reshape(-1)
            lo = int(math.floor(0.1 * mx))
            flat[w + 1] = lo                     # exactly 0.1 * max for 10 and 100: outside the box
            flat[npx - w - 2] = min(lo + 1, mx)  # the smallest value inside
            if f == 0:
                flat[npx - 1 - rng.integers(0, tail)] = mx          # the maximum only in the tail
            elif mx == 100:
                flat[0] = mx                                         # first pixel
            else:
                flat[npx - 1] = mx                                   # last pixel
    sky = rng.choice(np.array([0, 0, 0, 0, 1, 2, 128, 255], np.uint8), (NB, h, w))
    return segs, sky


@pytest.mark.parametrize('shared', [False, True], ids=['per_frame', 'shared'])
@pytest.mark.parametrize('wh', [(36, 21), (35, 19), (64, 48)], ids=['36x21', '35x19', '64x48'])
def test_graded_segmentation_and_sky(wh, shared):
    """Graded uint8 segmentation (0, 1, 126, 127, 128, 254, 255 and random values) with maxima 10, 30, 100, 1 and 0 at
    the first pixel, the last pixel or only in seg_max_kernel's tail, per-frame and shared (stride 0); 36 x 21 and
    35 x 19 give per-frame strides that are not multiples of 16 (the unaligned seg_max path) and 35 is not a multiple
    of 4 (VEC == 1).  Sky values other than 1.  Through residual_masks, detect (records) and detect_host."""
    import torch
    from mav_detection_b200 import engine
    from oracle import ccl_np
    from oracle import detect_np as dn
    w, h = wh
    rng = np.random.default_rng(w * 1000 + h + shared)
    segs, skys = _graded_frames(w, h, rng)
    if shared:
        segs = np.broadcast_to(segs[0], segs.shape).copy()
        skys = np.broadcast_to(skys[0], skys.shape).copy()
    ys, xs = np.mgrid[0:h, 0:w]
    flows = np.stack([np.stack([(xs - 0.4 * w) * 0.3, (ys - 0.45 * h) * 0.3], -1) + rng.normal(0, 0.8, (h, w, 2))
                      for _ in range(NB)]).astype(np.float32)
    gt = rng.normal(0, 2, (NB, h, w, 2)).astype(np.float32)
    ang = np.array([[0, 0, 0], [0.002, -0.001, 0.0005], [0, 0, 0], [0.001, 0.003, -0.002], [0.004, 0, 0.001],
                    [0, 0, 0]], np.float64)
    derot = [False, True, True, True, False, True]
    np.random.seed(31)
    samples = np.stack([np.concatenate(dn.draw_sample_indices(h, w)) for _ in range(NB)]).astype(np.int32)
    ref = []
    for f in range(NB):
        fi = 1 if derot[f] else 0
        fd, foe, phi, total, fixed = dn.frame_pipeline(fi, flows[f], ang[f], DT, skys[f] != 0, samples[f, :2000],
                                                       samples[f, 2000:], cr_arccos_f32=True)
        gd = dn.derotate(fi, gt[f], ang[f], DT)
        ref.append((fd, foe, total, fixed, gd))
    eng = _engine(w, h, NB)
    imu = engine.make_imu(NB, ang, DT, derotate=derot)
    seg_h, sky_h = (segs[0], skys[0]) if shared else (segs, skys)
    seg_d, sky_d = torch.from_numpy(np.ascontiguousarray(seg_h)).cuda(), torch.from_numpy(np.ascontiguousarray(sky_h)).cuda()
    flow_d = torch.from_numpy(flows).cuda()
    foe_d = torch.tensor(np.array([r[1] for r in ref]), dtype=torch.float64, device='cuda')
    _, tot, fix, st = eng.residual_masks(flow_d, imu, foe_d, sky=sky_d, seg=seg_d, want_phi=False)
    stats_rm = eng.stats_to_numpy(st)
    tot, fix = tot.cpu().numpy().astype(bool), fix.cpu().numpy().astype(bool)
    rec_d = eng.records_to_numpy(eng.detect(flow_d, imu, torch.from_numpy(samples).cuda(), sky=sky_d, seg=seg_d,
                                            gt_flow=torch.from_numpy(gt).cuda()))
    rec_h = eng.detect_host(flows, imu, samples, sky=np.ascontiguousarray(sky_h), seg=np.ascontiguousarray(seg_h),
                            gt_flow=gt).copy()
    for f in range(NB):
        fd, foe, total, fixed, gd = ref[f]
        seg = segs[f]
        assert seg.max() == SEG_MAXIMA[0 if shared else f]
        assert np.array_equal(tot[f], total) and np.array_equal(fix[f], fixed), f
        ct, cf = dn.metric_counts(seg, total), dn.metric_counts(seg, fixed)
        want = dict(n_total=total.sum(), n_fixed=fixed.sum(), positives=ct[0], negatives=ct[1], tp_total=ct[2],
                    fp_total=ct[3], tp_fixed=cf[2], fp_fixed=cf[3])
        box = dn.simple_bounding_box(seg)
        lab, comp = ccl_np.label(fixed)
        for src, s in (('residual_masks', stats_rm[f]), ('detect', rec_d[f]['stats']), ('detect_host', rec_h[f]['stats'])):
            for k in COUNT_KEYS:
                assert s[k] == want[k], (src, f, k, s[k], want[k])
            assert tuple(s['seg_bbox']) == box, (src, f, tuple(s['seg_bbox']), box)
            assert _sums_close(s['seg_flow_sum'], fd[seg > 127]), (src, f)
            if src != 'residual_masks':
                assert _sums_close(s['gt_flow_sum'], gd[seg > 127]), (src, f)
        for src, r in (('detect', rec_d[f]), ('detect_host', rec_h[f])):
            assert (r['foe'][0], r['foe'][1]) == foe, (src, f)
            assert r['n_labels'] == lab.max(), (src, f)
            k = min(32, comp.shape[0])
            assert np.array_equal(r['boxes'][:k], comp[:k]), (src, f)
    # the graded values matter: g >= 1 differs from g > 127 for the true positives, and the box threshold is not 128
    assert any(dn.metric_counts(segs[f], ref[f][3])[2] != int(((segs[f] > 127) & ref[f][3]).sum()) for f in range(NB))
    eng.close()


# ------------------------------------------------------------------------------------------------
# C. FoE and RANSAC thresholds
# ------------------------------------------------------------------------------------------------
FH, FW = 48, 64


def _gate_field(thr, dtype, rng, ry, rx):
    """Random flow whose sampled second points have magnitudes (in `dtype`) equal to the threshold's value in that
    precision, and one step below and above it."""
    f = rng.normal(0, 3, (FH, FW, 2)).astype(dtype)
    if not math.isfinite(thr) or thr > 1e20:
        return f, 0
    t = dtype(thr)
    vals = (np.nextafter(t, dtype(-np.inf)), t, np.nextafter(t, dtype(np.inf)))
    y2, x2 = ry[1000:], rx[1000:]
    for k in range(1000):
        v = vals[k % 3]
        s = 1 if (k // 3) % 2 else -1
        f[y2[k], x2[k]] = (s * v, 0) if (k // 6) % 2 else (0, s * v)
    mags = np.linalg.norm(f[y2, x2], axis=-1)
    return f, int((mags == t).sum())


MAG_THRESHOLDS = [2.5, 0.7, 0.0, 1e30, -1.0, NAN]


@pytest.mark.parametrize('thr', MAG_THRESHOLDS, ids=['2.5', '0.7', '0', '1e30', '-1', 'nan'])
def test_foe_magnitude_threshold(thr):
    """magnitude_threshold through foe (derotating with a zero rotation: float64 magnitudes of float32 flows; float32
    pass-through) and foe_dense (float32 and float64).  0.7 lies above its float32 value, so the float32 gate keeps
    second points a float64 comparison drops; 1e30 keeps nothing ((0, 0)); -1 and NaN keep everything."""
    import torch
    from mav_detection_b200 import engine
    from oracle import detect_np as dn
    rng = np.random.default_rng(5)
    np.random.seed(41)
    ry, rx = dn.draw_sample_indices(FH, FW)
    samples = torch.from_numpy(np.concatenate([ry, rx])[None].astype(np.int32)).cuda()
    f32, hits32 = _gate_field(thr, np.float32, rng, ry, rx)
    f64, hits64 = _gate_field(thr, np.float64, rng, ry, rx)
    if thr in (2.5, 0.7):
        assert hits32 > 100 and hits64 > 100
    eng = _engine(FW, FH)
    _set_params(eng, dict(magnitude_threshold=thr))
    cases = [('foe_dense f32', f32, dn.intersections(f32, ry, rx, thr), lambda: eng.foe_dense(torch.from_numpy(f32[None]).cuda(), samples)),
             ('foe_dense f64', f64, dn.intersections(f64, ry, rx, thr), lambda: eng.foe_dense(torch.from_numpy(f64[None]).cuda(), samples)),
             ('foe pass-through', f32, dn.intersections(f32, ry, rx, thr),
              lambda: eng.foe(torch.from_numpy(f32[None]).cuda(), engine.make_imu(1, derotate=False), samples)),
             ('foe derotating', f32, dn.intersections(dn.derotate(1, f32, np.zeros(3), DT), ry, rx, thr),
              lambda: eng.foe(torch.from_numpy(f32[None]).cuda(), engine.make_imu(1, derotate=True), samples))]
    for name, _, E, run in cases:
        foe, cnt = run()
        got = tuple(foe.cpu().numpy()[0])
        assert int(cnt[0]) == E.shape[0], (name, int(cnt[0]), E.shape[0])
        assert got == dn.ransac(E), (name, got, dn.ransac(E))
        if thr == 1e30:
            assert E.shape[0] == 0 and got == (0.0, 0.0)
    if thr == 0.7:
        # the float32 gate decides differently from a float64 one on this field: the count above is not vacuous
        assert dn.intersections(f32, ry, rx, thr).shape[0] != dn.intersections(f32.astype(np.float64), ry, rx, thr).shape[0]
    eng.close()


def _boundary_pairs(T, rng, n_angles=20000):
    """Points q around the centre c = T * (3.25, -1.5), classified by NumPy's distance |q - c| as ransac computes it
    (norm along the last axis): 'eq_lt' == T with dx^2 + dy^2 < T*T (what sqrt_threshold exists for), 'eq' == T
    otherwise, 'below' / 'above' one double either side.  Returns c and {class: [(angle in degrees, q)]}."""
    c = T * np.array([3.25, -1.5])
    out = {'eq_lt': [], 'eq': [], 'below': [], 'above': []}
    below, above = np.nextafter(T, 0.0), np.nextafter(T, np.inf)
    a = rng.uniform(0.0, 360.0, n_angles)
    q0 = c + T * np.stack([np.cos(np.radians(a)), np.sin(np.radians(a))], -1)
    for k in range(-4, 5):
        q = q0.copy()
        q[:, 1] += k * np.spacing(q0[:, 1])
        d = q - c
        dist = np.linalg.norm(d, axis=-1)
        s = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
        for name, sel in (('eq_lt', (dist == T) & (s < T * T)), ('eq', (dist == T) & ~(s < T * T)),
                          ('below', dist == below), ('above', dist == above)):
            out[name] += [(float(a[i]), q[i]) for i in np.flatnonzero(sel)]
    return c, out


def _ransac_sets(T, rng):
    """Estimate sets for a ransac threshold T.  For moderate T: group B (a centre and two points 0.25 T away, scores 2)
    first, then the centre c of _boundary_pairs with three points at NumPy distance exactly T and dx^2 + dy^2 < T*T,
    120 degrees apart, and partners at distance one double below T, one above and exactly T (with dx^2 + dy^2 >= T*T)
    in between.  c scores 1 and B wins; counting the exact-T pairs would give c 4.  Plus a random cloud with
    duplicates."""
    cloud = rng.normal(0, 40, (300, 2))
    cloud[100:110] = cloud[3] + rng.normal(0, 1, (10, 2))
    cloud[5] = cloud[3]
    sets = [cloud]
    if not (1e-6 < T < 1e6):
        return sets, None
    c, cls = _boundary_pairs(T, rng)

    def pick(name, near):
        cands = [q for a, q in cls[name] if min(abs(a - near), 360 - abs(a - near)) < 10]
        return [cands[0]] if cands else []

    far = c + np.array([0.0, 40.0 * T])
    E = [far, far + (0.25 * T, 0.0), far - (0.25 * T, 0.0), c]
    A = [pick('eq_lt', a) for a in (0.0, 120.0, 240.0)]
    if all(A):
        E += [q[0] for q in A]
    E += pick('below', 90.0) + pick('above', 200.0) + pick('eq', 310.0)
    sets.append(np.array(E))
    return sets, cls


RANSAC_THRESHOLDS = [30.0, 2.5, 0.1, 1 / 3, math.sqrt(2), 1e-3, 1e300, 0.0, -1.0, NAN, INF]


@pytest.mark.parametrize('T', RANSAC_THRESHOLDS, ids=['30', '2.5', '0.1', '1/3', 'sqrt2', '1e-3', '1e300', '0', '-1',
                                                       'nan', 'inf'])
def test_ransac_threshold(T):
    """ransac_threshold through ransac and foe_dense: sqrt(s) < T evaluated as s < s*, s* the smallest double whose
    square root is >= T.  For 2.5, 0.1, 1/3 and sqrt(2), s* < T*T; the sets hold pairs at NumPy distance exactly T with
    dx^2 + dy^2 < T*T, which must not count, and pairs one double inside and outside."""
    import torch
    from oracle import detect_np as dn
    rng = np.random.default_rng(7)
    sets, cls = _ransac_sets(T, rng)
    if T in (2.5, 0.1, 1 / 3, math.sqrt(2)):
        assert cls['eq_lt'] and cls['below'] and cls['above']
        # counting dx^2 + dy^2 < T*T instead would pick another estimate: the comparison below is not vacuous
        E = sets[1]
        assert E.shape[0] >= 7

        def ransac_sq(E):
            best, opt = (0.0, 0.0), 0
            for i in range(E.shape[0]):
                d = E - E[i]
                score = int(np.count_nonzero(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] < T * T)) - 1
                if score > opt:
                    opt, best = score, (float(E[i, 0]), float(E[i, 1]))
            return best
        assert ransac_sq(E) != dn.ransac(E, T)
    elif cls is not None:
        assert cls['eq'] and cls['below'] and cls['above']
    eng = _engine(FW, FH)
    for E in sets:
        got = tuple(eng.ransac(torch.from_numpy(np.ascontiguousarray(E)).cuda(), threshold=T).cpu().numpy())
        assert got == dn.ransac(E, T), (T, got, dn.ransac(E, T))
    # the same threshold through the FoE kernel (foe_dense on a float64 field)
    ys, xs = np.mgrid[0:FH, 0:FW]
    f = np.stack([(xs - 30.3) * 0.1, (ys - 20.7) * 0.1], -1) + rng.normal(0, 0.05, (FH, FW, 2))
    np.random.seed(43)
    ry, rx = dn.draw_sample_indices(FH, FW)
    _set_params(eng, dict(ransac_threshold=T))
    foe, cnt = eng.foe_dense(torch.from_numpy(f[None]).cuda(),
                             torch.from_numpy(np.concatenate([ry, rx])[None].astype(np.int32)).cuda())
    assert tuple(foe.cpu().numpy()[0]) == dn.foe_dense(f, ry, rx, 2.5, T)
    eng.close()


# ------------------------------------------------------------------------------------------------
# D. Graph replay keyed by the parameters
# ------------------------------------------------------------------------------------------------
def _graph_param_sets():
    sets = []
    for i in range(18):
        sets.append(dict(fixed_angle=5.0 + 2.5 * i, dyn_gain=4.0 + (i % 5), magnitude_threshold=1.0 + 0.5 * (i % 4),
                         ransac_threshold=10.0 + 5.0 * (i % 3), dyn_offset=0.25 if i % 6 else 20.0))
    return sets


def _records_equal(a, b):
    for k in ('foe', 'n_intersections', 'n_labels', 'boxes'):
        if not np.array_equal(a[k], b[k]):
            return False
    for k in COUNT_KEYS + ('max_phi', 'seg_bbox'):
        if not np.array_equal(a['stats'][k], b['stats'][k]):
            return False
    return True


def test_graph_replay_keyed_by_parameters():
    """One set of buffers, use_graph on, 18 parameter sets (more than the 16 graphs a handle keeps), then sets still
    cached and sets evicted: every call equals the direct launches (use_graph off) with the same parameters."""
    import torch
    from mav_detection_b200 import engine
    from oracle import detect_np as dn
    w, h, n = 96, 64, 2
    rng = np.random.default_rng(13)
    ys, xs = np.mgrid[0:h, 0:w]
    flows = np.stack([np.stack([(xs - 40.5) * 0.08, (ys - 30.2) * 0.08], -1) + rng.normal(0, 0.6, (h, w, 2))
                      for _ in range(n)]).astype(np.float32)
    np.random.seed(17)
    samples = np.stack([np.concatenate(dn.draw_sample_indices(h, w)) for _ in range(n)]).astype(np.int32)
    sky = np.zeros((h, w), np.uint8)
    sky[:6] = 1
    imu = engine.make_imu(n, np.array([[0.002, -0.001, 0.0005], [0, 0, 0]]), DT, derotate=[True, False])
    sets = _graph_param_sets()

    def run(eng, bufs, p):
        _set_params(eng, p)
        eng.detect(bufs['flow'], imu, bufs['samples'], sky=bufs['sky'], total_out=bufs['total'], fixed_out=bufs['fixed'],
                   records=bufs['records'])
        torch.cuda.synchronize()
        return (eng.records_to_numpy(bufs['records']).copy(), bufs['total'].cpu().numpy().copy(),
                bufs['fixed'].cpu().numpy().copy())

    def buffers():
        return dict(flow=torch.from_numpy(flows).cuda(), samples=torch.from_numpy(samples).cuda(),
                    sky=torch.from_numpy(sky).cuda(), total=torch.empty((n, h, w), dtype=torch.uint8, device='cuda'),
                    fixed=torch.empty((n, h, w), dtype=torch.uint8, device='cuda'),
                    records=torch.empty((n, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda'))

    eng_d = _engine(w, h, n)
    eng_d.set_tuning(use_graph=0)
    bd = buffers()
    direct = [run(eng_d, bd, p) for p in sets]
    eng_d.close()
    distinct = {(r[1].tobytes(), r[2].tobytes(), r[0]['foe'].tobytes()) for r in direct}
    assert len(distinct) >= 10
    assert all(not np.array_equal(direct[i][2], direct[i + 1][2]) for i in range(len(sets) - 1))
    eng_g = _engine(w, h, n)
    assert eng_g.get_tuning()['use_graph'] == 1
    bg = buffers()
    for i in list(range(len(sets))) + [17, 9, 2, 0, 1, 17]:
        rec, tot, fix = run(eng_g, bg, sets[i])
        for f in range(n):
            assert _records_equal(rec[f], direct[i][0][f]), (i, f)
        assert np.array_equal(tot, direct[i][1]) and np.array_equal(fix, direct[i][2]), i
    gs = eng_g.graph_stats()
    assert gs['direct'] == 0 and gs['captured'] == 16, gs
    eng_g.close()


# ------------------------------------------------------------------------------------------------
# E. Processor.run_detection honours its FocusOfExpansion's thresholds
# ------------------------------------------------------------------------------------------------
PROC_THRESHOLDS = dict(magnitude_threshold=0.1, ransac_threshold=2.5)


@pytest.mark.parametrize('who', ['own', 'other'])
@pytest.mark.parametrize('flow_source', ['dataset', 'farneback'])
def test_processor_uses_focus_of_expansion_thresholds(flow_source, who):
    """own: thresholds set on proc.focus_of_expansion after construction are the ones run_detection uses.  other: a
    second FocusOfExpansion on the same engine, with other thresholds and a get_FOE_dense call behind it, does not
    change the Processor's results."""
    import logging
    cv2 = pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, synth
    from mav_detection_b200.focus_of_expansion import FocusOfExpansion
    from mav_detection_b200.processor import Processor
    from mav_detection_b200.run_config import RunConfig
    from oracle import detect_np as dn
    W_, H_, F = 320, 240, 8
    p = dict(engine.SAMPLE_PARAMS)
    seq = synth.make_sequence(W_, H_, F, seq=2, with_rotation=True)
    cvflow = np.stack([cv2.calcOpticalFlowFarneback(seq.frames[i], seq.frames[i + 1], None, p['pyr_scale'], p['levels'],
                                                    p['winsize'], p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
                       for i in range(F - 1)])
    ds = synth.SyntheticDataset(seq, flows=cvflow)
    RunConfig.register_dataset(RunConfig.DatasetType.SIMULATION, lambda logger, sequence: ds)
    cfg = RunConfig(logging.getLogger('test'), 'simulation', 'synthetic', False, False, False, True, False, False,
                    'FLOW_FOE_CLUSTERING')
    proc = Processor(cfg, flow_source=flow_source, batch_frames=3, farneback_params=p, write_results=False)
    _set_params(proc.engine, {})            # the engine is shared: start from the defaults whatever ran before
    if who == 'own':
        proc.focus_of_expansion.magnitude_threshold = PROC_THRESHOLDS['magnitude_threshold']
        proc.focus_of_expansion.ransac_threshold = PROC_THRESHOLDS['ransac_threshold']
        expect = PROC_THRESHOLDS
    else:
        other = FocusOfExpansion(proc.detector.lucas_kanade, engine=proc.engine)
        other.magnitude_threshold = PROC_THRESHOLDS['magnitude_threshold']
        other.ransac_threshold = PROC_THRESHOLDS['ransac_threshold']
        other.get_FOE_dense(dn.derotate(1, cvflow[1], seq.omega[1], seq.dt))
        expect = dict(magnitude_threshold=2.5, ransac_threshold=30.0)
    np.random.seed(123)
    res = proc.run_detection()
    proc.release()
    assert sorted(res) == list(range(F - 1))
    np.random.seed(123)
    differs = 0
    for i in range(F - 1):
        ry, rx = dn.draw_sample_indices(H_, W_)
        if flow_source == 'dataset':
            flow = cvflow[i]
        else:
            eng = proc.engine
            flow = eng.farneback(torch.from_numpy(seq.frames[i:i + 2]).to(eng.device))[0].cpu().numpy()
        fd, foe, phi, total, fixed = dn.frame_pipeline(i, flow, seq.omega[i], seq.dt, seq.sky_mask, ry, rx,
                                                       cr_arccos_f32=True, **expect)
        alt = dn.foe_dense(fd, ry, rx, **{k: v for k, v in (PROC_THRESHOLDS if who == 'other' else
                                                            dict(magnitude_threshold=2.5, ransac_threshold=30.0)).items()})
        differs += alt != foe
        fr = res[i]
        assert fr.foe_dense == foe, (i, fr.foe_dense, foe)
        seg = seq.segmentation[i]
        assert (fr.tpr, fr.fpr, fr.tpr_fixed, fr.fpr_fixed) == dn.tpr_fpr(seg, total) + dn.tpr_fpr(seg, fixed), i
    assert differs >= 1          # the two threshold pairs lead to different FoEs: the test is not vacuous
