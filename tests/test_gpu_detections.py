"""GPU: per-frame detection tables (include/mavd.h: mavd_detection) against the NumPy oracle (tests/detections_np.py).

Labels, boxes, areas and index sums are exact.  flow_sum is a float64 sum accumulated with atomics, so it is compared
within 1e-12 x (the sum of the magnitudes of its terms) of NumPy's float64 sum of the same per-pixel values, which are
mavd_derotate's (the float32 flow widened for frames that do not derotate)."""
import ctypes as C
import logging

import numpy as np
import pytest

import detections_np as dnp

pytestmark = pytest.mark.gpu

SIZES = [(8, 8), (33, 17), (640, 480), (1920, 1080)]
MASKS = ['empty', 'single', 'noise1e-4', 'noise0.01', 'noise0.3', 'noise0.5', 'isolated', 'full', 'equal_area']
MAX_DETS = (1, 7, 32, 256)

_ENGINES = {}


def _engine(W, H, max_pairs=4):
    from mav_detection_b200 import engine
    key = (W, H, max_pairs)
    if key not in _ENGINES:
        _ENGINES[key] = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=max_pairs)
    return _ENGINES[key]


def _mask(kind, W, H, seed):
    rng = np.random.default_rng(seed)
    m = np.zeros((H, W), np.uint8)
    if kind == 'single':
        m[rng.integers(H), rng.integers(W)] = 1
    elif kind.startswith('noise'):
        m = (rng.random((H, W)) < float(kind[5:])).astype(np.uint8)
    elif kind == 'isolated':          # the most components a frame can hold under 8-connectivity
        m[::2, ::2] = 1
    elif kind == 'full':
        m[:] = 1
    elif kind == 'equal_area':        # 2 x 2 squares on a 3-pixel grid: every component has area 4
        for y in range(0, H - 1, 3):
            for x in range(0, W - 1, 3):
                m[y:y + 2, x:x + 2] = 1
        m[rng.random((H, W)) < 0.002] = 1
    return m


def _flow_and_imu(n, W, H, seed, derotate=None, zero_rot=None):
    from mav_detection_b200 import engine
    rng = np.random.default_rng(seed)
    flow = (rng.standard_normal((n, H, W, 2)) * 3).astype(np.float32)
    ang = rng.standard_normal((n, 3)) * 0.01
    if zero_rot is not None:
        ang[np.asarray(zero_rot, bool)] = 0.0
    der = [True] * n if derotate is None else derotate
    return flow, engine.make_imu(n, ang, 0.05, derotate=der)


def _derotated(eng, flow_t, imu):
    return eng.derotate(flow_t, imu).cpu().numpy()


def oracle(mask, fd, max_det=256):
    """The oracle's table and, with a flow, the sums of |term| of every flow_sum (the tolerance scale)."""
    ref = dnp.detections(mask, fd, max_det)
    return ref, (None if fd is None else dnp.detections(mask, np.abs(fd), max_det)['flow_sum'])


def check_table(got, mask, fd, max_det, where='', ref=None):
    """got: (max_det,) table of the GPU; mask (H, W); fd (H, W, 2) float64 per-pixel flow values or None.  ref: a
    precomputed oracle(mask, fd, k) with k >= max_det (the order is total: a shorter table is a prefix)."""
    ref, mag = ref if ref is not None else oracle(mask, fd, max_det)
    ref = ref[:max_det]
    for name in ('label', 'box', 'area', 'sum_x', 'sum_y'):
        assert np.array_equal(got[name], ref[name]), (where, name, got[name][:8], ref[name][:8])
    if fd is None:
        assert np.all(got['flow_sum'] == 0), where
        return
    mag = mag[:max_det]
    err = np.abs(got['flow_sum'] - ref['flow_sum'])
    assert np.all(err <= 1e-12 * mag), (where, float((err - 1e-12 * mag).max()))


def same_tables(a, b, where=''):
    """Two GPU tables of the same frame: integer fields bit-equal, flow sums to 1e-12 relative (atomic order)."""
    for name in ('label', 'box', 'area', 'sum_x', 'sum_y'):
        assert np.array_equal(a[name], b[name]), (where, name)
    assert np.allclose(a['flow_sum'], b['flow_sum'], rtol=1e-12, atol=1e-9), where


# ------------------------------------------------------------------------------------------------
# standalone mavd_detections against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('W,H', SIZES, ids=['%dx%d' % s for s in SIZES])
@pytest.mark.parametrize('kind', MASKS)
def test_standalone_matches_oracle(W, H, kind):
    import torch
    eng = _engine(W, H)
    masks = np.stack([_mask(kind, W, H, s) for s in (1, 2)])
    flow, imu = _flow_and_imu(2, W, H, seed=3, derotate=[True, False])
    flow_t = torch.from_numpy(flow).cuda()
    fd = _derotated(eng, flow_t, imu)
    mask_t = torch.from_numpy(masks).cuda()
    refs = [oracle(masks[f], fd[f]) for f in range(2)]
    for max_det in MAX_DETS:
        got = eng.detections_to_numpy(eng.detections(mask_t, flow_t, imu, max_det=max_det))
        nof = eng.detections_to_numpy(eng.detections(mask_t, max_det=max_det))
        for f in range(2):
            check_table(got[f], masks[f], fd[f], max_det, (kind, max_det, f), ref=refs[f])
            check_table(nof[f], masks[f], None, max_det, (kind, max_det, f, 'no flow'), ref=(refs[f][0], None))


@pytest.mark.parametrize('kind', ['noise0.3', 'equal_area', 'isolated'])
def test_standalone_misaligned_mask(kind):
    """A mask view one byte into its buffer takes the VEC=1 passes: same table as the aligned mask and the oracle."""
    import torch
    W, H = 640, 480
    eng = _engine(W, H)
    m = _mask(kind, W, H, 9)
    buf = torch.zeros(W * H + 1, dtype=torch.uint8, device='cuda')
    view = buf[1:].view(1, H, W)
    view.copy_(torch.from_numpy(m))
    aligned = torch.from_numpy(m).cuda().view(1, H, W)
    for max_det in (7, 256):
        got = eng.detections_to_numpy(eng.detections(view, max_det=max_det))[0]
        check_table(got, m, None, max_det, kind)
        same_tables(got, eng.detections_to_numpy(eng.detections(aligned, max_det=max_det))[0], kind)


def test_flow_sums_mix_derotation_modes():
    """One batch: a frame that does not derotate (float32 flow widened), one with a zero rotation, one rotating."""
    import torch
    W, H = 640, 480
    eng = _engine(W, H)
    masks = np.stack([_mask('noise0.3', W, H, s) for s in (4, 5, 6)])
    flow, imu = _flow_and_imu(3, W, H, seed=8, derotate=[False, True, True], zero_rot=[False, True, False])
    flow_t = torch.from_numpy(flow).cuda()
    fd = _derotated(eng, flow_t, imu)
    assert np.array_equal(fd[0], flow[0].astype(np.float64))
    got = eng.detections_to_numpy(eng.detections(torch.from_numpy(masks).cuda(), flow_t, imu, max_det=256))
    for f in range(3):
        check_table(got[f], masks[f], fd[f], 256, f)
    assert np.any(got[2]['flow_sum'] != got[1]['flow_sum'])


# ------------------------------------------------------------------------------------------------
# batch paths: *_det against *_ex, mavd_detections and the oracle
# ------------------------------------------------------------------------------------------------
def _rec(eng, r):
    return eng.records_to_numpy(r)


def _check_against_records(det, rec):
    for d in det:
        if d['label'] == 0 or d['label'] > 32:
            continue
        assert np.array_equal(rec['boxes'][d['label'] - 1], np.append(d['box'], d['area'])), d


def _process_det(eng, frames, imu, samples, n, flow, fixed, rec, max_det, det):
    from mav_detection_b200 import _lib
    _lib.check(eng.lib.mavd_process_det(eng._h, frames.data_ptr(), n, 1, imu, C.byref(eng.detect_params),
                                        samples.data_ptr(), C.byref(_lib.AuxInputs()), flow.data_ptr(), None,
                                        fixed.data_ptr(), rec.data_ptr(), max_det, det.data_ptr(), eng._stream()))


def _detect_det(eng, flow, imu, samples, n, fixed, rec, max_det, det):
    from mav_detection_b200 import _lib
    _lib.check(eng.lib.mavd_detect_det(eng._h, flow.data_ptr(), n, imu, C.byref(eng.detect_params), samples.data_ptr(),
                                       C.byref(_lib.AuxInputs()), None, fixed.data_ptr(), rec.data_ptr(), max_det,
                                       det.data_ptr(), eng._stream()))


def _table(eng, det, n, max_det):
    """The first n x max_det entries of a device buffer as (n, max_det) DETECTION_DTYPE."""
    from mav_detection_b200 import engine
    return det.view(-1)[:n * max_det * 56].view(n, max_det, 56).cpu().numpy().view(engine.DETECTION_DTYPE)[..., 0]


@pytest.mark.parametrize('motion', ['zoom', 'translate'])
def test_batch_paths_match_ex_calls_and_standalone(motion):
    """process_det / detect_det: records, masks and flow as the _ex calls; tables as mavd_detections on the returned
    estimate_fixed and flow, as the oracle, and as record.boxes for labels <= 32.  Every call twice (graph capture,
    then replay) into buffers poisoned before each run."""
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, F = 640, 480, 5
    n = F - 1
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    seq = synth.make_sequence(W, H, F, seq=7, with_rotation=True, motion=motion)
    frames = torch.from_numpy(seq.frames).cuda()
    samples = torch.from_numpy(sharded.draw_all_samples(n, H, W, seed=5)).cuda()
    imu = engine.make_imu(n, seq.omega[1:], seq.dt, derotate=[i >= 1 for i in range(n)])
    flow_ex = torch.empty((n, H, W, 2), dtype=torch.float32, device='cuda')
    fixed_ex = torch.empty((n, H, W), dtype=torch.uint8, device='cuda')
    rec_ex = _rec(eng, eng.process(frames, imu, samples, flow_out=flow_ex, fixed_out=fixed_ex))
    rec_dex = _rec(eng, eng.detect(flow_ex, imu, samples))
    flow = torch.empty_like(flow_ex)
    fixed = torch.empty_like(fixed_ex)
    rec_t = torch.empty((n, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    det_t = torch.empty((n, 256, 56), dtype=torch.uint8, device='cuda')
    fd = _derotated(eng, flow_ex, imu)
    fx = fixed_ex.cpu().numpy()
    refs = [oracle(fx[f], fd[f]) for f in range(n)]
    for max_det in (7, 256):
        for call in ('process', 'detect'):
            for run in range(2):                 # capture, then replay
                for t in (flow, fixed, rec_t, det_t):
                    t.view(torch.uint8).fill_(0xAB)
                if call == 'process':
                    _process_det(eng, frames, imu, samples, n, flow, fixed, rec_t, max_det, det_t)
                    assert torch.equal(flow, flow_ex)
                    assert sharded.compare_records(_rec(eng, rec_t), rec_ex) == [], (max_det, run)
                else:
                    _detect_det(eng, flow_ex, imu, samples, n, fixed, rec_t, max_det, det_t)
                    assert sharded.compare_records(_rec(eng, rec_t), rec_dex) == [], (max_det, run)
                assert torch.equal(fixed, fixed_ex)
                rec, det = _rec(eng, rec_t), _table(eng, det_t, n, max_det)
                alone = eng.detections_to_numpy(eng.detections(fixed_ex, flow_ex, imu, max_det=max_det))
                where = (call, max_det, run)
                for f in range(n):
                    same_tables(det[f], alone[f], where + (f,))
                    check_table(det[f], fx[f], fd[f], max_det, where + (f,), ref=refs[f])
                    _check_against_records(det[f], rec[f])
                    assert np.count_nonzero(det[f]['label']) == min(max_det, rec[f]['n_labels'])
    # the engine-level API returns the same tables
    rec2, det2 = eng.process(frames, imu, samples, detections=32)
    det2 = eng.detections_to_numpy(det2)
    rec3, det3 = eng.detect(flow_ex, imu, samples, detections=32)
    det3 = eng.detections_to_numpy(det3)
    for f in range(n):
        check_table(det2[f], fx[f], fd[f], 32, ('engine.process', f), ref=refs[f])
        check_table(det3[f], fx[f], fd[f], 32, ('engine.detect', f), ref=refs[f])
    gs = eng.graph_stats()
    assert gs['direct'] == 0 and gs['captured'] >= 6, gs
    eng.close()


def test_graph_keys_differ_in_max_det():
    """The same buffers with max_det 7 and then 32: two graphs, and each replay writes its own table size."""
    import torch
    from mav_detection_b200 import _lib, engine, sharded, synth
    W, H, n = 320, 240, 2
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    seq = synth.make_sequence(W, H, n + 1, seq=3, with_rotation=True, motion='translate')
    frames = torch.from_numpy(seq.frames).cuda()
    samples = torch.from_numpy(sharded.draw_all_samples(n, H, W, seed=1)).cuda()
    imu = engine.make_imu(n, seq.omega[1:], seq.dt)
    rec = torch.empty((n, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    fixed = torch.empty((n, H, W), dtype=torch.uint8, device='cuda')
    flow = torch.empty((n, H, W, 2), dtype=torch.float32, device='cuda')
    det = torch.empty((n, 32, engine.DETECTION_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    aux = _lib.AuxInputs()
    tables = {}
    for _ in range(2):
        for max_det in (7, 32):
            det.fill_(0xAB)
            _lib.check(eng.lib.mavd_process_det(eng._h, frames.data_ptr(), n, 1, imu, C.byref(eng.detect_params),
                                                samples.data_ptr(), C.byref(aux), flow.data_ptr(), None,
                                                fixed.data_ptr(), rec.data_ptr(), max_det, det.data_ptr(),
                                                eng._stream()))
            tables.setdefault(max_det, []).append(_table(eng, det, n, max_det))
    assert eng.graph_stats() == {'captured': 2, 'direct': 0}
    for f in range(n):
        same_tables(tables[7][0][f], tables[7][1][f])
        same_tables(tables[32][0][f], tables[32][1][f])
        same_tables(tables[7][0][f], tables[32][0][f][:7])
    eng.close()


# ------------------------------------------------------------------------------------------------
# batch invariance
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('pair_stride', [1, 2])
def test_tables_do_not_depend_on_the_batch(pair_stride):
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, N = 320, 240, 13
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=N)
    nf = N + 1 if pair_stride == 1 else 2 * N
    seq = synth.make_sequence(W, H, nf, seq=12, with_rotation=True, motion='translate')
    frames = torch.from_numpy(seq.frames).cuda()
    samples = sharded.draw_all_samples(N, H, W, seed=4)
    ang = seq.omega[1:1 + N] if seq.omega.shape[0] > N else np.zeros((N, 3))
    der = [i % 3 != 0 for i in range(N)]

    def run(first, n):
        fr = frames[first * pair_stride:first * pair_stride + (n + 1 if pair_stride == 1 else 2 * n)].contiguous()
        imu = engine.make_imu(n, ang[first:first + n], seq.dt, derotate=der[first:first + n])
        sm = torch.from_numpy(samples[first:first + n].copy()).cuda()
        _, det = eng.process(fr, imu, sm, pair_stride=pair_stride, detections=32)
        return eng.detections_to_numpy(det)

    alone = []
    for p in range(N):
        fr = frames[p * pair_stride:p * pair_stride + 2].contiguous()
        imu = engine.make_imu(1, ang[p:p + 1], seq.dt, derotate=der[p:p + 1])
        _, det = eng.process(fr, imu, torch.from_numpy(samples[p:p + 1].copy()).cuda(), pair_stride=2, detections=32)
        alone.append(eng.detections_to_numpy(det)[0])
    assert any(np.count_nonzero(a['label']) > 1 for a in alone)
    for bs in (13, 1, 5, 13):
        for first in range(0, N, bs):
            n = min(bs, N - first)
            got = run(first, n)
            for k in range(n):
                same_tables(got[k], alone[first + k], (bs, first + k))
    assert eng.graph_stats()['direct'] == 0
    eng.close()


# ------------------------------------------------------------------------------------------------
# host paths
# ------------------------------------------------------------------------------------------------
def _pinned(shape, dtype):
    import torch
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    return torch.empty((n,), dtype=torch.uint8, pin_memory=True).numpy().view(dtype).reshape(shape)


def test_host_calls_fill_the_tables():
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, n = 320, 240, 3
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    seq = synth.make_sequence(W, H, 3 * n + 3, seq=21, with_rotation=True, motion='translate')
    pb = eng.packed_mask_bytes
    jobs = []
    for slot in range(3):
        frames = seq.frames[slot * (n + 1):(slot + 1) * (n + 1)]
        bgr = _pinned(frames.shape + (3,), np.uint8)
        bgr[:] = frames[..., None]                        # gray replicated: cvtColor gives the same gray back
        samples = _pinned((n, 4000), np.int32)
        samples[:] = sharded.draw_all_samples(n, H, W, seed=slot)
        seg = eng.pack_mask_host(seq.segmentation[1:1 + n])
        imu = engine.make_imu(n, seq.omega[1:1 + n], seq.dt, derotate=[True, False, True])
        flow = _pinned((n, H, W, 2), np.float32)
        fixed = _pinned((n, pb), np.uint8)
        det = _pinned((n, 32), engine.DETECTION_DTYPE)
        det.view(np.uint8)[:] = 0xAB
        rec = eng.submit_host(slot, bgr, imu, samples, n_pairs=n, seg=seg, seg_packed=True, flow_out=flow,
                              fixed_out=fixed, fixed_packed=True, detections=det)
        jobs.append((slot, frames, imu, samples, flow, fixed, det, rec))
    for slot in (2, 0, 1):
        eng.wait_host(slot)
    for slot, frames, imu, samples, flow, fixed, det, rec in jobs:
        mask = eng.unpack_mask_host(fixed)
        flow_t = torch.from_numpy(flow.copy()).cuda()
        alone = eng.detections_to_numpy(eng.detections(torch.from_numpy(mask).cuda(), flow_t, imu, max_det=32))
        fd = _derotated(eng, flow_t, imu)
        for f in range(n):
            same_tables(det[f], alone[f], (slot, f))
            check_table(det[f], mask[f], fd[f], 32, (slot, f))
            _check_against_records(det[f], rec[f])
    # detect_host_det from the flow of the last batch
    slot, frames, imu, samples, flow, fixed, det, rec = jobs[-1]
    det2 = _pinned((n, 256), engine.DETECTION_DTYPE)
    fixed2 = np.empty((n, H, W), np.uint8)
    rec2 = eng.detect_host(flow, imu, samples, fixed_out=fixed2, detections=det2)
    fd = _derotated(eng, torch.from_numpy(flow.copy()).cuda(), imu)
    for f in range(n):
        check_table(det2[f], fixed2[f], fd[f], 256, ('detect_host', f))
        _check_against_records(det2[f], rec2[f])
    eng.close()


# ------------------------------------------------------------------------------------------------
# Processor
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('flow_source', ['dataset', 'farneback'])
def test_processor_detections(tmp_path, flow_source):
    import json
    import torch
    cv2 = pytest.importorskip('cv2')
    from mav_detection_b200 import engine, synth
    from mav_detection_b200.processor import Processor
    from mav_detection_b200.run_config import RunConfig
    from oracle import detect_np as dn
    W, H, F = 320, 240, 8
    p = dict(engine.SAMPLE_PARAMS)
    seq = synth.make_sequence(W, H, F, seq=2, with_rotation=True)
    cvflow = np.stack([cv2.calcOpticalFlowFarneback(seq.frames[i], seq.frames[i + 1], None, p['pyr_scale'], p['levels'],
                                                    p['winsize'], p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
                       for i in range(F - 1)])
    runs = {}
    for bf, md in ((4, 0), (1, 32), (4, 32)):
        out = tmp_path / ('r%d_%d' % (bf, md))
        ds = synth.SyntheticDataset(seq, flows=cvflow, results_path=str(out))
        RunConfig.register_dataset(RunConfig.DatasetType.SIMULATION, lambda logger, sequence: ds)
        cfg = RunConfig(logging.getLogger('test'), 'simulation', 'synthetic', False, False, False, True, False, False,
                        'FLOW_FOE_CLUSTERING')
        np.random.seed(99)
        proc = Processor(cfg, flow_source=flow_source, batch_frames=bf, farneback_params=p, max_detections=md)
        res = proc.run_detection()
        proc.release()
        runs[(bf, md)] = (res, proc.detections, out, proc.engine)
    base, _, base_dir, _ = runs[(4, 0)]
    assert runs[(4, 0)][1] == {}
    for key in ((1, 32), (4, 32)):
        res, dets, out, _ = runs[key]
        assert sorted(dets) == list(range(F - 1))
        for i in range(F - 1):
            a, b = res[i], base[i]
            assert (a.foe_dense, a.tpr, a.fpr, a.tpr_fixed, a.fpr_fixed, a.drone_size_pixels, a.time) == \
                (b.foe_dense, b.tpr, b.fpr, b.tpr_fixed, b.fpr_fixed, b.drone_size_pixels, b.time), (key, i)
            assert np.allclose(a.drone_flow_pixels, b.drone_flow_pixels, rtol=1e-12, atol=0, equal_nan=True), (key, i)
            ja = json.load(open(out / ('image_%05d.json' % i)))
            jb = json.load(open(base_dir / ('image_%05d.json' % i)))
            fa, fb = ja.pop('drone_flow_pixels', None), jb.pop('drone_flow_pixels', None)
            assert json.dumps(ja, sort_keys=True) == json.dumps(jb, sort_keys=True), (key, i)
            assert np.allclose(np.asarray(fa, float), np.asarray(fb, float), rtol=1e-12, atol=0, equal_nan=True)
    d1, d4 = runs[(1, 32)][1], runs[(4, 32)][1]
    for i in range(F - 1):
        assert [(d.label, d.box, d.area, d.centroid) for d in d1[i]] == [(d.label, d.box, d.area, d.centroid) for d in d4[i]]
        for x, y in zip(d1[i], d4[i]):
            assert np.allclose(x.flow, y.flow, rtol=1e-12, atol=1e-12)
    # the chained oracle with the same global random stream (test_gpu_api.test_processor_run_detection_matches_oracle_chain)
    np.random.seed(99)
    np.random.randint(20, H - 20, 1000); np.random.randint(20, W - 20, 1000)
    n = 2000 + 2000 // 3
    np.random.randint(0, 255, (n, 3)); np.random.randint(0, 255, (n, 3)); np.random.randint(0, n, n)
    eng = runs[(4, 32)][3]
    for i in range(F - 1):
        ry, rx = dn.draw_sample_indices(H, W)
        flow = cvflow[i] if flow_source == 'dataset' else \
            eng.farneback(torch.from_numpy(seq.frames[i:i + 2]).to(eng.device))[0].cpu().numpy()
        fd, foe, phi, total, fixed = dn.frame_pipeline(i, flow, seq.omega[i], seq.dt, seq.sky_mask, ry, rx,
                                                       cr_arccos_f32=True)
        fd = fd.astype(np.float64)
        ref = dnp.detections(fixed, fd, 32)
        mag = dnp.detections(fixed, np.abs(fd), 32)['flow_sum']
        got = d4[i]
        assert len(got) == np.count_nonzero(ref['label']), i
        for d, r, m in zip(got, ref, mag):
            assert (d.label, d.box, d.area) == (r['label'], tuple(r['box']), r['area'])
            assert d.centroid == (r['sum_x'] / r['area'], r['sum_y'] / r['area'])
            assert np.all(np.abs(np.asarray(d.flow) * d.area - r['flow_sum']) <= 1e-12 * m + 1e-300)


# ------------------------------------------------------------------------------------------------
# errors and workspace
# ------------------------------------------------------------------------------------------------
def test_rejected_arguments_and_lazy_workspace():
    import torch
    from mav_detection_b200 import _lib, engine, sharded, synth
    W, H = 64, 48
    quiet = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=2)
    ws_quiet = quiet.workspace_bytes
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=2)
    assert eng.workspace_bytes == ws_quiet
    mask = torch.zeros((1, H, W), dtype=torch.uint8, device='cuda')
    flow = torch.zeros((1, H, W, 2), dtype=torch.float32, device='cuda')
    for bad in (0, 257, -1):
        with pytest.raises(ValueError):
            eng.detections(mask, max_det=bad)
    det = torch.empty((1, 256, 56), dtype=torch.uint8, device='cuda')
    imu = engine.make_imu(1)
    lib = eng.lib
    for md in (0, 257):
        with pytest.raises(ValueError):
            _lib.check(lib.mavd_detections(eng._h, mask.data_ptr(), 1, None, None, md, det.data_ptr(), eng._stream()))
    with pytest.raises(ValueError):          # NULL table
        _lib.check(lib.mavd_detections(eng._h, mask.data_ptr(), 1, None, None, 8, None, eng._stream()))
    with pytest.raises(ValueError):          # a flow without an imu array
        _lib.check(lib.mavd_detections(eng._h, mask.data_ptr(), 1, flow.data_ptr(), None, 8, det.data_ptr(),
                                       eng._stream()))
    seq = synth.make_sequence(W, H, 2, seq=1)
    frames = torch.from_numpy(seq.frames).cuda()
    samples = torch.from_numpy(sharded.draw_all_samples(1, H, W, seed=0)).cuda()
    rec = torch.empty((1, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    aux = _lib.AuxInputs()
    for md in (0, 257):
        with pytest.raises(ValueError):
            _lib.check(lib.mavd_process_det(eng._h, frames.data_ptr(), 1, 1, imu, None, samples.data_ptr(),
                                            C.byref(aux), None, None, None, rec.data_ptr(), md, det.data_ptr(),
                                            eng._stream()))
        with pytest.raises(ValueError):
            _lib.check(lib.mavd_detect_det(eng._h, flow.data_ptr(), 1, imu, None, samples.data_ptr(), C.byref(aux),
                                           None, None, rec.data_ptr(), md, det.data_ptr(), eng._stream()))
        with pytest.raises(ValueError):
            eng.process(frames, imu, samples, detections=md)
    with pytest.raises(ValueError):
        eng.detect_host(np.zeros((1, H, W, 2), np.float32), imu, samples.cpu().numpy(),
                        detections=np.zeros((1, 300), engine.DETECTION_DTYPE))
    with pytest.raises(ValueError):
        eng.detect_host(np.zeros((1, H, W, 2), np.float32), imu, samples.cpu().numpy(),
                        detections=np.zeros((1, 8), np.int64))
    assert eng.workspace_bytes == ws_quiet            # rejected calls allocate nothing
    eng.detections(mask, max_det=8)
    torch.cuda.synchronize()
    assert eng.workspace_bytes > ws_quiet
    assert quiet.workspace_bytes == ws_quiet          # a handle that never asked keeps its footprint
    quiet.process(frames, imu, samples)
    torch.cuda.synchronize()
    assert quiet.workspace_bytes == ws_quiet
    quiet.close()
    eng.close()
