"""GPU: a pair's results do not depend on the batch, the buffer offsets or the host slot that carry it.

A frame pair's flow, masks and record are a function of its two frames, its IMU entry, its sample indices and its sky and
segmentation masks only: sharded runs, Processor.run_detection at any batch_frames and bench.py --dump-outputs A/B
comparisons all rely on it.  The library, though, chooses kernels, grids and launch counts per call: pairs are grouped
by IT_PAIR_GROUP = 4 (the last group may be short), the iteration tile height follows tiles x pairs, the pyramid sweep's
band count follows words x frames, alignment decides the word / vec4 / TMA paths, a batch mixing float32-frame and
derotating pairs makes two residual launches, graphs are cached by key (which frames derotate is read from the device
copy of the imu data at replay time) and three host slots overlap their copies with the compute.

The reference for "alone" is the same pair run with n_pairs=1, pair_stride=2 from a freshly allocated tensor on the
same engine.  The tilings are bit-identical by design (DESIGN §4: the sums are re-seeded at rows = 0 mod 8), so every
comparison below is exact; the record comparison is sharded.compare_records, which allows 1e-12 on the two float64
flow sums only (they are accumulated with atomics).  Every call runs twice with graphs on (capture, then replay), the
outputs poisoned before each run, and the batches of a test share one engine in the order large -> small -> large, so
that scratch left by a larger batch is present when a smaller one runs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPE_MEAN_TOL = 1e-3      # flow against cv2.calcOpticalFlowFarneback: the bar of test_gpu_farneback.py


def _samples(n, H, W, seed):
    from mav_detection_b200 import sharded
    return sharded.draw_all_samples(n, H, W, seed=seed)


def _offset_buffer(shape, dtype, offset):
    """An empty CUDA tensor that starts `offset` bytes into a larger buffer (offset 0: a fresh, aligned tensor)."""
    import torch
    if offset == 0:
        return torch.empty(shape, dtype=dtype, device='cuda')
    nb = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    buf = torch.zeros(nb + offset, dtype=torch.uint8, device='cuda')
    return buf[offset:offset + nb].view(dtype).reshape(shape)


def _offset_copy(t, offset):
    """A CUDA copy of t that starts `offset` bytes into a larger buffer (as test_gpu_detect_params.py)."""
    view = _offset_buffer(tuple(t.shape), t.dtype, offset)
    view.copy_(t)
    return view


def _no_direct_launches(eng):
    gs = eng.graph_stats()
    assert gs['captured'] >= 1 and gs['direct'] == 0, gs


def _max_diff(a, b):
    return float((a.double() - b.double()).abs().max())


# ------------------------------------------------------------------------------------------------
# 1. Farneback: batch size, pair stride, position in the sequence and alignment
# ------------------------------------------------------------------------------------------------
def _alone_flows(eng, frames):
    """Flow of every pair (i, i + 1) of `frames`, each run as n_pairs=1, pair_stride=2 from a fresh tensor."""
    import torch
    out = []
    for i in range(frames.shape[0] - 1):
        t = torch.from_numpy(np.ascontiguousarray(frames[i:i + 2])).to(eng.device)
        flow = torch.empty((1, eng.height, eng.width, 2), dtype=torch.float32, device=eng.device)
        got = []
        for _ in range(2):
            flow.fill_(float('nan'))
            eng.farneback(t, n_pairs=1, pair_stride=2, out=flow)
            got.append(flow[0].clone())
        assert torch.equal(got[0], got[1]), i
        out.append(got[0])
    return torch.stack(out)


def _run_batch(eng, frames_t, n, stride, out):
    """The batch twice (graph capture, then replay) into `out`; both runs must write the same flow."""
    import torch
    got = []
    for _ in range(2):
        out.fill_(float('nan'))
        eng.farneback(frames_t, n_pairs=n, pair_stride=stride, out=out)
        got.append(out.clone())
    assert torch.equal(got[0], got[1]), (n, stride, 'replay differs from capture')
    return got[0]


def _check_pairs(flow, alone, first, n, stride, where):
    import torch
    for p in range(n):
        a = first + (p if stride == 1 else 2 * p)
        assert torch.equal(flow[p], alone[a]), where + ('pair', p, 'frames', a, _max_diff(flow[p], alone[a]))


def _farneback_invariance(W, H, params, ns, align_ns, cv2_pairs, seq_id, offsets=(0, 1, 3)):
    cv2 = pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, synth
    nmax = max(ns)
    n_frames = max(offsets) + 2 * nmax + 1          # one frame more than the longest batch reads
    seq = synth.make_sequence(W, H, n_frames, seq=seq_id)
    eng = engine.Engine(W, H, params, max_pairs=nmax)
    assert eng.get_tuning()['use_graph'] == 1
    frames_d = torch.from_numpy(seq.frames).to(eng.device)
    alone = _alone_flows(eng, seq.frames)
    for i in cv2_pairs:
        ref = cv2.calcOpticalFlowFarneback(seq.frames[i], seq.frames[i + 1], None, params['pyr_scale'], params['levels'],
                                           params['winsize'], params['iterations'], params['poly_n'],
                                           params['poly_sigma'], params['flags'])
        epe = np.linalg.norm(alone[i].cpu().numpy() - ref, axis=-1).mean()
        assert epe < EPE_MEAN_TOL, (i, epe)
    out = torch.empty((nmax, H, W, 2), dtype=torch.float32, device=eng.device)
    for n in ns:
        for stride in (1, 2):
            for k in offsets:
                # frames[k:] moves the base pointer by k * W * H bytes and is longer than the batch needs
                flow = _run_batch(eng, frames_d[k:], n, stride, out[:n])
                _check_pairs(flow, alone, k, n, stride, ('n', n, 'stride', stride, 'offset', k))
    for n in align_ns:
        for off in (1, 2, 4, 8, 16):
            for flow_off in (0, 8):
                frames_t = _offset_copy(frames_d[:n + 1], off)
                assert frames_t.data_ptr() % 16 == off % 16
                fl = _offset_buffer((n, H, W, 2), torch.float32, flow_off)
                if flow_off:
                    assert fl.data_ptr() % 16 == 8            # float2-aligned, not 16-byte aligned
                flow = _run_batch(eng, frames_t, n, 1, fl)
                _check_pairs(flow, alone, 0, n, 1, ('n', n, 'frame byte offset', off, 'flow byte offset', flow_off))
    _no_direct_launches(eng)
    eng.close()


# 1, 2, 3, 4, 5, 7, 8, 9, 12, 13 pairs: every remainder of the pair groups of 4, the 64 x 16 / 64 x 32 tile switch at
# n = 2 (level 0) and n = 11 (level 1), several groups; ordered large -> small -> large
NS_640 = (13, 9, 5, 3, 1, 2, 4, 7, 8, 12)


@pytest.mark.parametrize('size', [(640, 480), (328, 200), (333, 257)], ids=['640x480', '328x200', '333x257'])
def test_farneback_pairs_equal_their_alone_runs(size):
    """640 x 480: everything aligned.  328 x 200: W % 16 = 8, level-0 polyexp runs without TMA.  333 x 257: odd, no
    word loads in the pyramid (no sweep), no 16-byte flow stores.  Batch sizes, both pair strides, the batch taken at
    offsets 0, 1 and 3 into a longer sequence, frames at byte offsets 1, 2, 4, 8 and 16 and the flow at byte offset 8:
    every pair equals the same pair run alone, bit for bit."""
    from mav_detection_b200 import engine
    W, H = size
    if size == (640, 480):
        _farneback_invariance(W, H, engine.SAMPLE_PARAMS, NS_640, (9, 1, 5), (0, 7, 15), seq_id=51)
    elif size == (328, 200):
        _farneback_invariance(W, H, engine.SAMPLE_PARAMS, (9, 5, 1, 2, 4, 13), (5, 1), (2, 11), seq_id=52)
    else:
        _farneback_invariance(W, H, engine.SAMPLE_PARAMS, (9, 3, 1, 2, 5), (5, 1), (1, 8), seq_id=53)


@pytest.mark.parametrize('window', ['gauss15', 'box21'])
def test_farneback_window_variants_equal_their_alone_runs(window):
    """A Gaussian window (flags=256, winsize 15: the TMA kernel) and a winsize-21 box window (the generic iter_kernel on
    its 3-D grid) at 1, 5 and 9 pairs."""
    from mav_detection_b200 import engine
    p = dict(engine.SAMPLE_PARAMS)
    if window == 'gauss15':
        p['flags'] = 256
    else:
        p['winsize'] = 21
    _farneback_invariance(640, 480, p, (9, 1, 5), (5,), (0, 6), seq_id=54 if window == 'gauss15' else 55,
                          offsets=(0, 1))


# ------------------------------------------------------------------------------------------------
# 2. Detection: float32-frame, zero-rotation and rotating frames in one batch
# ------------------------------------------------------------------------------------------------
DW, DH, DN = 320, 240, 5
# F: derotate = 0 (the float32 frame, MODE 1); Z: derotate = 1 with a zero rotation (MODE 0, no-rotation build);
# R: derotate = 1 with a non-zero rotation.  [Z,R] and [R,Z] have the same graph key: the second replays the first's
# graph with other imu contents.
COMPOSITIONS = ('R', 'ZZ', 'FR', 'FZ', 'ZR', 'RZ', 'FZR', 'RZFRZ')


def _kind_imu(kinds, ang, dt):
    from mav_detection_b200 import engine
    a = np.array([np.zeros(3) if k == 'Z' else ang[j] for j, k in enumerate(kinds)])
    return engine.make_imu(len(kinds), a, dt, derotate=[k != 'F' for k in kinds])


def _oracle_frame(flow, kind, ang, dt, sky, seg, smp):
    """The chained oracle of one frame: dn.frame_pipeline (float32 frame for F, float64 derotation otherwise) and the
    labelling oracle on its fixed mask."""
    from oracle import ccl_np
    from oracle import detect_np as dn
    a = np.zeros(3) if kind == 'Z' else ang
    fd, foe, phi, total, fixed = dn.frame_pipeline(0 if kind == 'F' else 1, flow, a, dt, sky != 0, smp[:2000],
                                                   smp[2000:], cr_arccos_f32=True)
    lab, stats = ccl_np.label(fixed.astype(np.uint8))
    return dict(fd=fd, foe=foe, phi=phi, total=total, fixed=fixed, n_labels=lab.max(), boxes=stats[:32], seg=seg)


def _check_oracle(where, rec, fixed, total, ref, kind):
    from oracle import detect_np as dn
    seg = ref['seg']
    assert tuple(rec['foe']) == ref['foe'], where + ('foe', tuple(rec['foe']), ref['foe'])
    assert np.array_equal(fixed.astype(bool), ref['fixed']), where + ('fixed', int((fixed.astype(bool) != ref['fixed']).sum()))
    if total is not None:
        assert np.array_equal(total.astype(bool), ref['total']), where + ('total',)
    st = rec['stats']
    ct, cf = dn.metric_counts(seg, ref['total']), dn.metric_counts(seg, ref['fixed'])
    assert (st['n_total'], st['n_fixed']) == (ref['total'].sum(), ref['fixed'].sum()), where
    assert (st['positives'], st['negatives'], st['tp_total'], st['fp_total'], st['tp_fixed'], st['fp_fixed']) == \
        (ct[0], ct[1], ct[2], ct[3], cf[2], cf[3]), where
    assert tuple(st['seg_bbox']) == dn.simple_bounding_box(seg), where
    assert np.allclose(st['seg_flow_sum'], ref['fd'][seg > 127].astype(np.float64).sum(axis=0), rtol=1e-9), where
    assert rec['n_labels'] == ref['n_labels'], where
    k = min(32, ref['boxes'].shape[0])
    assert np.array_equal(rec['boxes'][:k], ref['boxes'][:k]), where
    # the float32 pre-decision (FAST) runs for the derotating frames under the default parameters: no max phi there
    if kind == 'F':
        assert st['max_phi'] == float(ref['phi'].max()) and st['max_phi'] != -1.0, where
    else:
        assert st['max_phi'] == -1.0, where


def test_detection_mixed_frame_kinds_in_one_batch():
    """Batches mixing F, Z and R frames through detect and process (total mask requested or not), detect_host,
    per-frame and shared sky / segmentation, aligned and misaligned buffers (VEC == 1): every frame's record, fixed mask
    and total mask equal the frame run alone and the chained oracle, and max_phi is -1 exactly for the derotated
    frames (FAST) and never for F frames.  The device buffers of a batch size are reused from call to call, so
    compositions with the same key ([Z,R], [R,Z]) replay one graph."""
    pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, sharded, synth
    seq = synth.make_sequence(DW, DH, DN + 1, seq=56, with_rotation=True)
    dt = seq.dt
    ang = np.array([seq.omega[j + 1] * (1.0 + 0.5 * j) for j in range(DN)])
    samples = _samples(DN, DH, DW, 57)
    sky_per = np.zeros((DN, DH, DW), np.uint8)
    for j in range(DN):
        sky_per[j, :6 + 4 * j] = 1
        sky_per[j, 6 + 4 * j, ::3] = 255
    sky_shared = np.zeros((DH, DW), np.uint8)
    sky_shared[:10] = 1
    seg_per = np.ascontiguousarray(seq.segmentation[1:DN + 1])
    seg_shared = np.ascontiguousarray(seq.segmentation[1])
    eng = engine.Engine(DW, DH, engine.SAMPLE_PARAMS, max_pairs=DN)
    frames_d = torch.from_numpy(seq.frames).to(eng.device)
    flows_d = eng.farneback(frames_d).clone()           # flows with a real FoE: the detection masks are not empty
    flows = flows_d.cpu().numpy()
    samples_d = torch.from_numpy(samples).to(eng.device)

    def masks(shared, j):
        return (sky_shared, seg_shared) if shared else (sky_per[j], seg_per[j])

    # the oracle and the alone run of frame j as kind k (one n = 1 buffer set for all of them)
    oracle, alone = {}, {}
    one = dict(flow=torch.empty((1, DH, DW, 2), dtype=torch.float32, device=eng.device),
               smp=torch.empty((1, samples.shape[1]), dtype=torch.int32, device=eng.device),
               sky=torch.empty((1, DH, DW), dtype=torch.uint8, device=eng.device),
               seg=torch.empty((1, DH, DW), dtype=torch.uint8, device=eng.device),
               total=torch.empty((1, DH, DW), dtype=torch.uint8, device=eng.device),
               fixed=torch.empty((1, DH, DW), dtype=torch.uint8, device=eng.device),
               rec=torch.empty((1, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device=eng.device))

    def reference(j, kind, shared):
        key = (j, kind, shared)
        if key not in alone:
            sky, seg = masks(shared, j)
            oracle[key] = _oracle_frame(flows[j], kind, ang[j], dt, sky, seg, samples[j])
            one['flow'].copy_(flows_d[j:j + 1])
            one['smp'].copy_(samples_d[j:j + 1])
            one['sky'][0].copy_(torch.from_numpy(sky))
            one['seg'][0].copy_(torch.from_numpy(seg))
            got = []
            for _ in range(2):
                one['total'].fill_(7)
                one['fixed'].fill_(7)
                one['rec'].fill_(0xAB)
                eng.detect(one['flow'], _kind_imu(kind, ang[j:j + 1], dt), one['smp'], sky=one['sky'], seg=one['seg'],
                           total_out=one['total'], fixed_out=one['fixed'], records=one['rec'])
                got.append((eng.records_to_numpy(one['rec']), one['fixed'][0].cpu().numpy(), one['total'][0].cpu().numpy()))
            assert sharded.compare_records(got[0][0], got[1][0]) == [] and np.array_equal(got[0][1], got[1][1]), key
            alone[key] = got[0]
            _check_oracle(('alone',) + key, got[0][0][0], got[0][1], got[0][2], oracle[key], kind)
            assert got[0][1].any(), key                 # non-trivial masks
        return alone[key], oracle[key]

    bufs = {}

    def device_buffers(api, n, aligned, shared):
        key = (api, n, aligned, shared)
        if key not in bufs:
            mo = 0 if aligned else 1
            shp = (DH, DW) if shared else (n, DH, DW)
            bufs[key] = dict(flow=_offset_buffer((n, DH, DW, 2), torch.float32, 0 if aligned else 8),
                             sky=_offset_buffer(shp, torch.uint8, mo), seg=_offset_buffer(shp, torch.uint8, mo),
                             total=_offset_buffer((n, DH, DW), torch.uint8, mo),
                             fixed=_offset_buffer((n, DH, DW), torch.uint8, mo),
                             smp=torch.empty((n, samples.shape[1]), dtype=torch.int32, device=eng.device),
                             rec=torch.empty((n, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device=eng.device))
        return bufs[key]

    def run_device(api, kinds, aligned, shared, with_total):
        n = len(kinds)
        b = device_buffers(api, n, aligned, shared)
        if not aligned:
            assert b['flow'].data_ptr() % 16 == 8 and b['seg'].data_ptr() % 4 == 1 and b['fixed'].data_ptr() % 4 == 1
        sky, seg = (sky_shared, seg_shared) if shared else (sky_per[:n], seg_per[:n])
        b['sky'].copy_(torch.from_numpy(np.ascontiguousarray(sky)))
        b['seg'].copy_(torch.from_numpy(np.ascontiguousarray(seg)))
        b['smp'].copy_(samples_d[:n])
        imu = _kind_imu(kinds, ang[:n], dt)
        total = b['total'] if with_total else None
        out = []
        for _ in range(2):
            b['total'].fill_(7)
            b['fixed'].fill_(7)
            b['rec'].fill_(0xAB)
            if api == 'detect':
                b['flow'].copy_(flows_d[:n])
                eng.detect(b['flow'], imu, b['smp'], sky=b['sky'], seg=b['seg'], total_out=total, fixed_out=b['fixed'],
                           records=b['rec'])
            else:
                b['flow'].fill_(float('nan'))
                eng.process(frames_d, imu, b['smp'], n_pairs=n, sky=b['sky'], seg=b['seg'], flow_out=b['flow'],
                            total_out=total, fixed_out=b['fixed'], records=b['rec'])
                assert torch.equal(b['flow'], flows_d[:n]), (api, kinds, aligned, shared)
            out.append((eng.records_to_numpy(b['rec']), b['fixed'].cpu().numpy(),
                        b['total'].cpu().numpy() if with_total else None))
        return out

    def run_host(kinds, shared):
        n = len(kinds)
        sky, seg = (sky_shared, seg_shared) if shared else (sky_per[:n], seg_per[:n])
        out = []
        for _ in range(2):
            fixed = np.full((n, DH, DW), 7, np.uint8)
            rec = eng.detect_host(np.ascontiguousarray(flows[:n]), _kind_imu(kinds, ang[:n], dt),
                                  np.ascontiguousarray(samples[:n]), sky=np.ascontiguousarray(sky),
                                  seg=np.ascontiguousarray(seg), fixed_out=fixed).copy()
            out.append((rec, fixed, None))
        return out

    for shared in (False, True):
        for kinds in COMPOSITIONS:
            for j, k in enumerate(kinds):
                reference(j, k, shared)
    variants = [('host', True, shared, False) for shared in (False, True)] + \
        [(api, aligned, shared, with_total) for api in ('detect', 'process') for aligned in (True, False)
         for shared in (False, True) for with_total in (True, False)]
    for api, aligned, shared, with_total in variants:
        for kinds in COMPOSITIONS:
            before = eng.graph_stats()['captured']
            runs = run_host(kinds, shared) if api == 'host' else run_device(api, kinds, aligned, shared, with_total)
            if kinds == 'RZ' and before < 16:
                assert eng.graph_stats()['captured'] == before, 'RZ did not replay the graph of ZR'
            for t, (rec, fixed, total) in enumerate(runs):
                for j, k in enumerate(kinds):
                    where = (api, 'aligned' if aligned else 'offset', 'shared' if shared else 'per-frame',
                             'total' if with_total else 'no total', kinds, 'run', t, 'frame', j, k)
                    (arec, afix, atot), ref = reference(j, k, shared)
                    assert sharded.compare_records(rec[j:j + 1], arec) == [], where + \
                        tuple(sharded.compare_records(rec[j:j + 1], arec))
                    assert np.array_equal(fixed[j], afix), where + ('fixed', int((fixed[j] != afix).sum()))
                    if total is not None:
                        assert np.array_equal(total[j], atot), where + ('total', int((total[j] != atot).sum()))
                    if t == 0:
                        _check_oracle(where, rec[j], fixed[j], total[j] if total is not None else None, ref, k)
    _no_direct_launches(eng)
    eng.close()


# ------------------------------------------------------------------------------------------------
# 3. The sharded cut on one GPU
# ------------------------------------------------------------------------------------------------
def test_sequence_cut_at_every_point_equals_one_batch():
    """13 pairs at 640 x 480 as one process batch, then cut into [0, c) + [c, 13) for every c and into the
    shard_range shares of 2, 3 and 4 ranks: flows, fixed masks and records bit-equal.  The derotate flag and the IMU
    entry of a pair follow its global index, its sample rows come from draw_all_samples sliced per shard."""
    pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, N = 640, 480, 13
    seq = synth.make_sequence(W, H, N + 1, seq=58, with_rotation=True)
    samples = sharded.draw_all_samples(N, H, W, seed=59)
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=N)
    dev = eng.device
    frames = torch.from_numpy(seq.frames).to(dev)
    smp = torch.from_numpy(samples).to(dev)
    seg = torch.from_numpy(np.ascontiguousarray(seq.segmentation)).to(dev)
    flow = torch.empty((N, H, W, 2), dtype=torch.float32, device=dev)
    fixed = torch.empty((N, H, W), dtype=torch.uint8, device=dev)
    rec = torch.empty((N, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)

    def run(parts):
        got = []
        for _ in range(2):
            flow.fill_(float('nan'))
            fixed.fill_(7)
            rec.fill_(0xAB)
            for lo, hi in parts:
                if hi == lo:
                    continue
                n = hi - lo
                imu = engine.make_imu(n, seq.omega[lo + 1:hi + 1], seq.dt, derotate=[lo + i >= 1 for i in range(n)])
                eng.process(frames[lo:], imu, smp[lo:hi], n_pairs=n, seg=seg[lo + 1:hi + 1], flow_out=flow[lo:hi],
                            fixed_out=fixed[lo:hi], records=rec[lo:hi])
            got.append((flow.clone(), fixed.clone(), eng.records_to_numpy(rec)))
        return got

    (ref_flow, ref_fixed, ref_rec), again = run([(0, N)])
    assert torch.equal(again[0], ref_flow) and torch.equal(again[1], ref_fixed)
    assert sharded.compare_records(again[2], ref_rec) == []
    assert ref_fixed.any()
    # the whole batch is right, not just consistent: two pairs against cv2 and the chained oracle
    import cv2
    from oracle import ccl_np
    from oracle import detect_np as dn
    p = engine.SAMPLE_PARAMS
    for i in (0, 9):
        f = ref_flow[i].cpu().numpy()
        cvf = cv2.calcOpticalFlowFarneback(seq.frames[i], seq.frames[i + 1], None, p['pyr_scale'], p['levels'],
                                           p['winsize'], p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
        assert np.linalg.norm(f - cvf, axis=-1).mean() < EPE_MEAN_TOL, i
        fd, foe, phi, total, fix = dn.frame_pipeline(i, f, seq.omega[i + 1], seq.dt, seq.sky_mask, samples[i, :2000],
                                                     samples[i, 2000:], cr_arccos_f32=True)
        assert tuple(ref_rec[i]['foe']) == foe and np.array_equal(ref_fixed[i].cpu().numpy().astype(bool), fix), i
        lab, _ = ccl_np.label(fix.astype(np.uint8))
        assert ref_rec[i]['n_labels'] == lab.max(), i
    cuts = [[(0, c), (c, N)] for c in range(1, N)]
    cuts += [[sharded.shard_range(N, world, r) for r in range(world)] for world in (2, 3, 4)]
    for parts in cuts:
        for t, (fl, fx, rc) in enumerate(run(parts)):
            where = (parts, 'run', t)
            assert torch.equal(fl, ref_flow), where + ('flow', _max_diff(fl, ref_flow))
            assert torch.equal(fx, ref_fixed), where + ('fixed',)
            assert sharded.compare_records(rc, ref_rec) == [], where + tuple(sharded.compare_records(rc, ref_rec))
    _no_direct_launches(eng)
    eng.close()


# ------------------------------------------------------------------------------------------------
# 4. Three host slots in flight
# ------------------------------------------------------------------------------------------------
HW, HH, HN = 320, 240, 5
# per slot: frame format, batch, pair stride, frame kinds (cycled), masks, outputs
HOST_SLOTS = {
    0: dict(bgr=False, n=5, stride=1, kinds='FRZRR', packed=False, shared_sky=False, flow_out=True, gt=False),
    1: dict(bgr=True, n=3, stride=2, kinds='RRF', packed=True, shared_sky=False, flow_out=False, gt=True),
    2: dict(bgr=False, n=1, stride=1, kinds='R', packed=False, shared_sky=True, flow_out=False, gt=False),
}


class _HostBatch:
    """One submission's inputs and outputs in pinned host memory (pageable memory would serialise the copies), and
    the device-buffer reference call that must give the same outputs."""

    def __init__(self, eng, seq, slot, n, stride, seed, keep):
        import cv2
        import torch
        from mav_detection_b200 import engine
        spec = HOST_SLOTS[slot]
        self.eng, self.slot, self.n, self.stride, self.spec = eng, slot, n, stride, spec
        rng = np.random.default_rng(seed)
        need = n + 1 if stride == 1 else 2 * n
        start = int(rng.integers(0, seq.frames.shape[0] - need + 1))

        def pinned(shape, dtype):
            dtype = np.dtype(dtype)
            t = torch.empty((max(int(np.prod(shape)) * dtype.itemsize, 1),), dtype=torch.uint8, pin_memory=True)
            keep.append(t)
            return t.numpy()[:int(np.prod(shape)) * dtype.itemsize].view(dtype).reshape(shape)

        gray = seq.frames[start:start + need]
        if spec['bgr']:
            tint = rng.integers(0, 40, gray.shape + (3,)).astype(np.int16)
            bgr = np.clip(gray[..., None].astype(np.int16) + tint - 20, 0, 255).astype(np.uint8)
            self.frames = pinned(bgr.shape, np.uint8)
            self.frames[:] = bgr
            self.gray = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr])
        else:
            self.frames = pinned(gray.shape, np.uint8)
            self.frames[:] = gray
            self.gray = gray
        second = [start + (i + 1 if stride == 1 else 2 * i + 1) for i in range(n)]      # the later frame of each pair
        kinds = (spec['kinds'] * HN)[:n]
        ang = np.array([np.zeros(3) if k == 'Z' else seq.omega[s] * (1.0 + 0.3 * (s % 4)) for k, s in zip(kinds, second)])
        self.imu_args = (n, ang, seq.dt, [k != 'F' for k in kinds])
        self.samples = pinned((n, 4000), np.int32)
        self.samples[:] = _samples(n, HH, HW, seed)
        if spec['shared_sky']:
            self.sky = np.zeros((HH, HW), np.uint8)
            self.sky[:4 + start % 20] = 1
        else:
            self.sky = np.zeros((n, HH, HW), np.uint8)
            for i, s in enumerate(second):
                self.sky[i, :4 + s % 20] = 1
        self.seg = np.ascontiguousarray(seq.segmentation[second])
        if spec['packed']:
            self.sky_in, self.seg_in = pinned(self.sky.shape[:-2] + (eng.packed_mask_bytes,), np.uint8), \
                pinned((n, eng.packed_mask_bytes), np.uint8)
            self.sky_in[:] = eng.pack_mask_host(self.sky)
            self.seg_in[:] = eng.pack_mask_host(self.seg)
        else:
            self.sky_in, self.seg_in = pinned(self.sky.shape, np.uint8), pinned(self.seg.shape, np.uint8)
            self.sky_in[:] = self.sky
            self.seg_in[:] = self.seg
        self.gt = None
        if spec['gt']:
            self.gt = pinned((n, HH, HW, 2), np.float32)
            self.gt[:] = rng.normal(0, 2, (n, HH, HW, 2))
        self.records = pinned((n,), engine.RECORD_DTYPE)
        self.records.view(np.uint8)[:] = 0xAB
        self.fixed = pinned((n, eng.packed_mask_bytes) if spec['packed'] else (n, HH, HW), np.uint8)
        self.fixed[:] = 7
        self.flow = None
        if spec['flow_out']:
            self.flow = pinned((n, HH, HW, 2), np.float32)
            self.flow[:] = np.nan
        self.key = (slot, n, stride, kinds)

    def submit(self):
        from mav_detection_b200 import engine
        self.eng.submit_host(self.slot, self.frames, engine.make_imu(*self.imu_args), self.samples, n_pairs=self.n,
                             pair_stride=self.stride, sky=self.sky_in, seg=self.seg_in, flow_out=self.flow,
                             fixed_out=self.fixed, records=self.records, gt_flow=self.gt, seg_packed=self.spec['packed'],
                             sky_packed=self.spec['packed'], fixed_packed=self.spec['packed'])

    def check(self, where):
        """After wait_host(slot): the outputs equal eng.process on device buffers (run now, with other slots in flight
        on the same stream)."""
        import torch
        from mav_detection_b200 import engine, sharded
        eng, n = self.eng, self.n
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(eng.device)
        flow = torch.empty((n, HH, HW, 2), dtype=torch.float32, device=eng.device)
        fixed = torch.empty((n, HH, HW), dtype=torch.uint8, device=eng.device)
        rec = eng.process(d(self.gray), engine.make_imu(*self.imu_args), d(self.samples), n_pairs=n,
                          pair_stride=self.stride, sky=d(self.sky), seg=d(self.seg), flow_out=flow, fixed_out=fixed,
                          gt_flow=None if self.gt is None else d(self.gt))
        rec, fixed = eng.records_to_numpy(rec), fixed.cpu().numpy()
        where = where + self.key
        assert sharded.compare_records(self.records, rec) == [], where + tuple(sharded.compare_records(self.records, rec))
        got = eng.unpack_mask_host(self.fixed) if self.spec['packed'] else self.fixed
        assert np.array_equal(got, fixed), where + ('fixed', int((got != fixed).sum()))
        assert fixed.any(), where
        if self.flow is not None:
            assert np.array_equal(self.flow, flow.cpu().numpy()), where + ('flow',)
        if self.gt is not None:
            assert np.abs(rec['stats']['gt_flow_sum']).sum() > 0, where


def test_three_host_slots_in_flight():
    """submit_host on all three slots before any wait (gray / BGR frames, byte / packed masks, per-frame / shared sky,
    flow_out / packed fixed / ground-truth flow on some slots only), waits out of order and resubmissions while another
    slot is in flight, two full rotations (capture and replay with other slots in flight), then a pass over 24 distinct
    keys, more than the 16 graphs the handle keeps, with three batches in flight."""
    pytest.importorskip('cv2')
    from mav_detection_b200 import synth
    from mav_detection_b200 import engine
    seq = synth.make_sequence(HW, HH, 16, seq=60, with_rotation=True)
    eng = engine.Engine(HW, HH, engine.SAMPLE_PARAMS, max_pairs=HN)
    keep = []

    def batch(slot, seed, n=None, stride=None):
        spec = HOST_SLOTS[slot]
        return _HostBatch(eng, seq, slot, n or spec['n'], stride or spec['stride'], seed, keep)

    live = {s: batch(s, 100 + s) for s in (0, 1, 2)}
    for s in (0, 1, 2):
        live[s].submit()
    for r in (1, 2):
        eng.wait_host(2)
        eng.wait_host(0)
        for s in (2, 0):
            live[s].check(('rotation', r - 1))
            live[s] = batch(s, 100 + 10 * r + s)
            live[s].submit()
        eng.wait_host(1)
        live[1].check(('rotation', r - 1))
        live[1] = batch(1, 100 + 10 * r + 1)
        live[1].submit()
    for s in (2, 0, 1):
        eng.wait_host(s)
        live[s].check(('rotation', 2))
    # more distinct keys than the graph cache holds, cycled with three batches in flight
    plans = {0: [(5, 1), (4, 2), (3, 1), (2, 2), (1, 1), (5, 2), (4, 1), (3, 2)],
             1: [(3, 2), (2, 1), (1, 2), (3, 1), (2, 2), (1, 1), (4, 2), (5, 1)],
             2: [(1, 1), (2, 1), (3, 2), (4, 1), (5, 2), (1, 2), (2, 2), (3, 1)]}
    inflight, keys = {}, set()
    for k in range(24):
        s = k % 3
        if s in inflight:
            eng.wait_host(s)
            inflight.pop(s).check(('lru', k))
        n, stride = plans[s][k // 3]
        b = batch(s, 200 + k, n, stride)
        keys.add(b.key)
        b.submit()
        inflight[s] = b
    for s in sorted(inflight):
        eng.wait_host(s)
        inflight[s].check(('lru', 'drain'))
    assert len(keys) > 16
    _no_direct_launches(eng)
    eng.close()


# ------------------------------------------------------------------------------------------------
# 5. Processor batch sizes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('flow_source', ['farneback', 'farneback-bgr'])
def test_processor_results_do_not_depend_on_batch_frames(flow_source):
    """Processor.run_detection on a 12-frame sequence (11 pairs) with batch_frames 1, 2, 4 and 5 (three batches through
    the slots, the last with one pair): identical FrameResults, and equal to the chained oracle for batch_frames 4.
    drone_flow_pixels is the float64 atomic flow sum over positives: compared to 1e-12 as sharded.compare_records."""
    import logging
    import torch
    cv2 = pytest.importorskip('cv2')
    from mav_detection_b200 import engine, synth
    from mav_detection_b200.processor import Processor
    from mav_detection_b200.run_config import RunConfig
    from oracle import detect_np as dn
    W, H, F = 320, 240, 12
    params = dict(engine.SAMPLE_PARAMS)
    seq = synth.make_sequence(W, H, F, seq=61, with_rotation=True)
    bgr = flow_source.endswith('-bgr')
    results, engines = {}, {}
    for bf in (1, 2, 4, 5):
        ds = synth.SyntheticDataset(seq, bgr=bgr)
        RunConfig.register_dataset(RunConfig.DatasetType.SIMULATION, lambda logger, sequence: ds)
        cfg = RunConfig(logging.getLogger('test'), 'simulation', 'synthetic', False, False, False, True, False, False,
                        'FLOW_FOE_CLUSTERING')
        np.random.seed(99)
        proc = Processor(cfg, flow_source='farneback', batch_frames=bf, farneback_params=params, write_results=False)
        results[bf] = proc.run_detection()
        engines[bf] = proc.engine
        proc.release()
        assert sorted(results[bf]) == list(range(F - 1)), bf
    ref = results[4]
    for bf in (1, 2, 5):
        for i in range(F - 1):
            a, b = results[bf][i], ref[i]
            where = (bf, i)
            assert a.foe_dense == b.foe_dense, where
            assert (a.tpr, a.fpr, a.tpr_fixed, a.fpr_fixed) == (b.tpr, b.fpr, b.tpr_fixed, b.fpr_fixed), where
            assert np.allclose(a.drone_flow_pixels, b.drone_flow_pixels, rtol=1e-12, atol=0), where
            assert (a.drone_size_pixels, a.center_phi, a.time, a.foe_gt) == \
                (b.drone_size_pixels, b.center_phi, b.time, b.foe_gt), where
    # the oracle with the same global random stream (test_gpu_api.test_processor_run_detection_matches_oracle_chain)
    np.random.seed(99)
    np.random.randint(20, H - 20, 1000); np.random.randint(20, W - 20, 1000)
    n = 2000 + 2000 // 3
    np.random.randint(0, 255, (n, 3)); np.random.randint(0, 255, (n, 3)); np.random.randint(0, n, n)
    eng = engines[4]
    p = params
    for i in range(F - 1):
        ry, rx = dn.draw_sample_indices(H, W)
        flow = eng.farneback(torch.from_numpy(seq.frames[i:i + 2]).to(eng.device))[0].cpu().numpy()
        if i in (0, 10):
            cvf = cv2.calcOpticalFlowFarneback(seq.frames[i], seq.frames[i + 1], None, p['pyr_scale'], p['levels'],
                                               p['winsize'], p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
            assert np.linalg.norm(flow - cvf, axis=-1).mean() < EPE_MEAN_TOL, i
        fd, foe, phi, total, fixed = dn.frame_pipeline(i, flow, seq.omega[i], seq.dt, seq.sky_mask, ry, rx,
                                                       cr_arccos_f32=True)
        fr = ref[i]
        assert fr.foe_dense == foe, (i, fr.foe_dense, foe)
        seg = seq.segmentation[i]
        assert (fr.tpr, fr.fpr, fr.tpr_fixed, fr.fpr_fixed) == dn.tpr_fpr(seg, total) + dn.tpr_fpr(seg, fixed), i
        assert fr.drone_size_pixels == int((seg > 127).sum())
        assert np.allclose(fr.drone_flow_pixels, fd[seg > 127].astype(np.float64).mean(axis=0), rtol=1e-9, atol=1e-12)
