"""Frame streams (include/mavd.h: mavd_stream_start): a handle keeps each stream's last frame expanded on the device and
pairs it with the next frame of that stream.  A step must equal, bit for bit, the pair_stride 2 call on the explicit
(previous, new) frames: flow, records, total / fixed masks and detection tables (whose float64 flow sums are summed
with atomics and compared to 1e-12, as sharded.compare_records does).  The explicit reference runs on a second engine
with the same parameters, because any non-stream Farneback call on a handle ends its streams."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPE_MEAN_TOL = 1e-3      # flow against cv2.calcOpticalFlowFarneback: the bar of test_gpu_farneback.py
MAX_DET = 8


# ------------------------------------------------------------------------------------------------
# CPU: the new prototypes
# ------------------------------------------------------------------------------------------------
def test_stream_prototypes_match_the_header():
    from mav_detection_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'mavd.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    decls = dict((name, args) for name, args in
                 re.findall(r'\bint\s+(mavd_stream_[a-z_]+)\s*\(([^;{]*?)\)\s*;', src, flags=re.S))
    assert sorted(decls) == ['mavd_stream_farneback', 'mavd_stream_process', 'mavd_stream_start',
                             'mavd_stream_submit_host']
    ctype = {'mavd_handle': C.c_void_p, 'int32_t': C.c_int32, 'const mavd_imu*': C.POINTER(_lib.Imu),
             'const mavd_detect_params*': C.POINTER(_lib.DetectParams),
             'const mavd_aux_inputs*': C.POINTER(_lib.AuxInputs)}
    for name, args in decls.items():
        res, argtypes = _lib.SIGNATURES[name]
        assert res is C.c_int, name
        params = [a.strip() for a in args.split(',')]
        assert len(params) == len(argtypes), name
        for p, t in zip(params, argtypes):
            typ = p.rsplit(' ', 1)[0].replace(' *', '*')
            assert t is ctype.get(typ, C.c_void_p), (name, p, t)     # everything else is a pointer
    # each step takes its counterpart's arguments after pair_stride, in the same order
    for stream, plain, cut in (('mavd_stream_process', 'mavd_process', 4), ('mavd_stream_submit_host',
                                                                           'mavd_submit_host', 5)):
        assert _lib.SIGNATURES[stream][1][cut:] == _lib.SIGNATURES[plain][1][cut:], stream


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def _frames(W, H, n, seq):
    from mav_detection_b200 import synth
    if W < 64 or H < 48:                 # below synth's moving blob: noise frames
        return np.random.default_rng(seq).integers(0, 256, (n, H, W), dtype=np.uint8)
    return synth.make_sequence(W, H, n, seq=seq).frames


class Cameras:
    """n_streams independent frame sequences; next(s) hands out camera s's next frame."""

    def __init__(self, W, H, n_streams, n_frames, seed=0):
        self.seqs = [_frames(W, H, n_frames, seed + s) for s in range(n_streams)]
        self.pos = [0] * n_streams

    def next(self, s):
        f = self.seqs[s][self.pos[s]]
        self.pos[s] += 1
        return f


def _imu(n, seed):
    from mav_detection_b200 import engine
    rng = np.random.default_rng(seed)
    return engine.make_imu(n, ang=rng.normal(0, 2e-3, (n, 3)), dt=0.05)


def _det_equal(a, b):
    from mav_detection_b200.engine import Engine
    a, b = Engine.detections_to_numpy(a), Engine.detections_to_numpy(b)
    for name in ('label', 'box', 'area', 'sum_x', 'sum_y'):
        if not np.array_equal(a[name], b[name]):
            return False
    return np.allclose(a['flow_sum'], b['flow_sum'], rtol=1e-12, atol=1e-9)


def _process_outputs(eng, n):
    import torch
    H, W = eng.height, eng.width
    return dict(flow_out=torch.full((n, H, W, 2), float('nan'), device=eng.device),
                total_out=torch.full((n, H, W), 7, dtype=torch.uint8, device=eng.device),
                fixed_out=torch.full((n, H, W), 7, dtype=torch.uint8, device=eng.device))


def _explicit(ref, prev, new, imu, samples):
    """mavd_process with pair_stride 2 on the explicit pairs (prev[i], new[i])."""
    import torch
    n = len(new)
    frames = torch.from_numpy(np.stack([f for pair in zip(prev, new) for f in pair])).to(ref.device)
    out = _process_outputs(ref, n)
    rec, det = ref.process(frames, imu, samples, n_pairs=n, pair_stride=2, detections=MAX_DET, **out)
    return dict(out, records=rec, det=det)


def _step(eng, ids, new, imu, samples):
    import torch
    out = _process_outputs(eng, len(ids))
    rec, det = eng.stream_process(torch.from_numpy(np.stack(new)).to(eng.device), ids, imu, samples,
                                  detections=MAX_DET, **out)
    return dict(out, records=rec, det=det)


def _assert_same(got, want, where):
    import torch
    from mav_detection_b200 import sharded
    from mav_detection_b200.engine import Engine
    for k in ('flow_out', 'total_out', 'fixed_out'):
        assert torch.equal(got[k], want[k]), (where, k)
    bad = sharded.compare_records(Engine.records_to_numpy(got['records']), Engine.records_to_numpy(want['records']))
    assert not bad, (where, bad)
    assert _det_equal(got['det'], want['det']), where


class Runner:
    """Drives a stream engine and its explicit reference over a schedule and checks every step."""

    def __init__(self, W, H, params, max_pairs, n_frames, seed=0, tuning=None):
        import torch
        from mav_detection_b200 import engine, sharded
        self.eng = engine.Engine(W, H, params, max_pairs=max_pairs)
        self.ref = engine.Engine(W, H, params, max_pairs=max_pairs)
        if tuning:
            self.eng.set_tuning(**tuning)
            self.ref.set_tuning(**tuning)
        self.cams = Cameras(W, H, max_pairs, n_frames, seed)
        self.kept = {}
        self.samples = torch.from_numpy(sharded.draw_all_samples(max_pairs, H, W, seed=seed)).to(self.eng.device)
        self.n_steps = 0

    def start(self, ids):
        import torch
        new = [self.cams.next(s) for s in ids]
        self.eng.stream_start(torch.from_numpy(np.stack(new)).to(self.eng.device), ids)
        self.kept.update(zip(ids, new))

    def step(self, ids, check=True):
        new = [self.cams.next(s) for s in ids]
        imu = _imu(len(ids), self.n_steps)
        samples = self.samples[:len(ids)]
        got = _step(self.eng, ids, new, imu, samples)
        if check:
            want = _explicit(self.ref, [self.kept[s] for s in ids], new, imu, samples)
            _assert_same(got, want, ('step', self.n_steps, 'ids', ids))
        self.kept.update(zip(ids, new))
        self.n_steps += 1
        return got

    def close(self):
        self.eng.close()
        self.ref.close()


# ------------------------------------------------------------------------------------------------
# 1. + 2. bit equality over sizes and parameters, stream patterns
# ------------------------------------------------------------------------------------------------
def _params(name):
    from mav_detection_b200 import engine
    s = engine.SAMPLE_PARAMS
    return {'sample': s, 'pyr04': dict(s, pyr_scale=0.4), 'reference': engine.REFERENCE_PARAMS,
            'gauss': dict(s, flags=256), 'w21': dict(s, winsize=21), 'gauss_w21': dict(s, flags=256, winsize=21),
            'poly7': dict(s, poly_n=7, poly_sigma=1.5), 'poly6': dict(s, poly_n=6, poly_sigma=1.3),
            'iter1': dict(s, iterations=1), 'c4': dict(s, levels=7, iterations=10)}[name]


# every table-addressed kernel variant is launched by one of these: the generic iteration with box and Gaussian windows
# (winsize 21), the expansion with poly_n 5, 7, 8 and a run-time poly_n (6), with and without TMA staging (W % 16 != 0
# at 333 x 257), and the level-entry matrices with every coordinate mode (power-of-two, float64 at pyr_scale 0.4, the
# host tables through mavd_tuning.mat_coord = 1)


# every pattern: all ids in order, permuted, a strict subset (streams 0 and 2 skip a step, then resume against their own
# kept frame), a restart by stream_start, n = 1 and n = max_pairs
PATTERN = [('start', [0, 1, 2, 3]), ('step', [0, 1, 2, 3]), ('step', [2, 0, 3, 1]), ('step', [1, 3]),
           ('step', [0, 2, 1]), ('start', [3]), ('step', [3]), ('step', [1, 0, 3, 2])]


@pytest.mark.gpu
@pytest.mark.parametrize('W,H,params', [
    (8, 8, 'sample'), (333, 257, 'sample'), (640, 480, 'sample'), (640, 480, 'pyr04'), (640, 480, 'reference'),
    (640, 480, 'gauss'), (640, 480, 'w21'), (640, 480, 'gauss_w21'), (640, 480, 'poly7'), (640, 480, 'poly6'),
    (640, 480, 'iter1'), (640, 480, 'tables'), (1920, 1080, 'sample')])
def test_stream_steps_equal_explicit_pairs(W, H, params):
    tuning = {'mat_coord': 1} if params == 'tables' else None
    r = Runner(W, H, _params('sample' if params == 'tables' else params), 4, 8, seed=W + H, tuning=tuning)
    for kind, ids in PATTERN:
        r.start(ids) if kind == 'start' else r.step(ids)
    r.close()


@pytest.mark.gpu
def test_one_4k_step_equals_its_explicit_pair():
    r = Runner(3840, 2160, _params('c4'), 2, 2, seed=4)
    r.start([1, 0])
    r.step([0, 1])
    r.close()


@pytest.mark.gpu
def test_stream_farneback_equals_pair_stride_2_and_cv2():
    cv2 = pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine
    W, H, p = 640, 480, engine.SAMPLE_PARAMS
    eng, ref = engine.Engine(W, H, p, max_pairs=3), engine.Engine(W, H, p, max_pairs=3)
    cams = Cameras(W, H, 3, 4, seed=7)
    kept = [cams.next(s) for s in range(3)]
    eng.stream_start(torch.from_numpy(np.stack(kept[::-1])).to(eng.device), [2, 1, 0])
    for ids in ([0, 1, 2], [1], [2, 0, 1]):
        new = [cams.next(s) for s in ids]
        flow = eng.stream_farneback(torch.from_numpy(np.stack(new)).to(eng.device), ids)
        pairs = torch.from_numpy(np.stack([f for s, n in zip(ids, new) for f in (kept[s], n)])).to(ref.device)
        want = ref.farneback(pairs, n_pairs=len(ids), pair_stride=2)
        assert torch.equal(flow, want), ids
        for i, s in enumerate(ids):
            cvf = cv2.calcOpticalFlowFarneback(kept[s], new[i], None, p['pyr_scale'], p['levels'], p['winsize'],
                                               p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
            assert np.linalg.norm(flow[i].cpu().numpy() - cvf, axis=-1).mean() < EPE_MEAN_TOL, (ids, s)
            kept[s] = new[i]
    # taps read the last non-stream call: refused after a stream call, available again after a non-stream one
    with pytest.raises(ValueError, match='stream'):
        eng.tap('R', 0, 0)
    eng.farneback(pairs, n_pairs=1, pair_stride=2)
    assert eng.tap('R', 0, 0).shape == (H, W, 5)
    eng.close()
    ref.close()


# ------------------------------------------------------------------------------------------------
# 3. rejections leave the streams as they were
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejected_calls_change_no_stream():
    import torch
    from mav_detection_b200 import _lib
    r = Runner(320, 240, _params('sample'), 3, 24, seed=3)
    eng, lib = r.eng, r.eng.lib
    frames = torch.zeros((3, 240, 320), dtype=torch.uint8, device=eng.device)
    flow = torch.empty((4, 240, 320, 2), device=eng.device)
    r.start([0, 2])

    def rejected(ids, n=None, match=None):
        arr = (C.c_int32 * max(1, len(ids)))(*ids)
        rc = lib.mavd_stream_farneback(eng._h, frames.data_ptr(), len(ids) if n is None else n, arr, flow.data_ptr(),
                                       None)
        assert rc == _lib.MAVD_ERR_INVALID, ids
        msg = lib.mavd_last_error().decode()
        if match:
            assert re.search(match, msg), msg
        r.step([2, 0])                      # the streams are where they were

    rejected([0, 0], match='stream 0 appears twice')
    rejected([-1], match='outside')
    rejected([3], match='outside')
    rejected([0, 1], match='stream 1 is not started')
    rejected([0, 2, 1, 1], n=4, match='exceeds max_pairs')
    assert lib.mavd_stream_farneback(eng._h, None, 1, (C.c_int32 * 1)(0), flow.data_ptr(), None) == _lib.MAVD_ERR_INVALID
    assert lib.mavd_stream_farneback(eng._h, frames.data_ptr(), 1, None, flow.data_ptr(), None) == _lib.MAVD_ERR_INVALID
    assert lib.mavd_stream_start(eng._h, frames.data_ptr(), 2, (C.c_int32 * 2)(1, 1), None) == _lib.MAVD_ERR_INVALID
    r.step([0, 2])
    # a NULL ids array is rejected by every stream call, whatever n (never taken for a pair call)
    imu1 = _imu(1, 0)
    rec_d = torch.empty((1, np.dtype(_lib.FrameRecord).itemsize), dtype=torch.uint8, device=eng.device)
    samples_h = np.ascontiguousarray(r.samples[:1].cpu().numpy())
    host_frames = np.zeros((1, 240, 320), np.uint8)
    host_recs = np.empty((1,), dtype=np.dtype(_lib.FrameRecord))
    for n in (0, 1):
        calls = {
            'stream_start': lambda: lib.mavd_stream_start(eng._h, frames.data_ptr(), n, None, None),
            'stream_farneback': lambda: lib.mavd_stream_farneback(eng._h, frames.data_ptr(), n, None, flow.data_ptr(),
                                                                  None),
            'stream_process': lambda: lib.mavd_stream_process(eng._h, frames.data_ptr(), n, None, imu1, None,
                                                              r.samples.data_ptr(), None, flow.data_ptr(), None, None,
                                                              rec_d.data_ptr(), 0, None, None),
            'stream_submit_host': lambda: lib.mavd_stream_submit_host(eng._h, 0, host_frames.ctypes.data, n, None, imu1,
                                                                      None, samples_h.ctypes.data, None, 0, None, None,
                                                                      host_recs.ctypes.data, 0, None, None)}
        for name, call in calls.items():
            assert call() == _lib.MAVD_ERR_INVALID, (name, n)
            assert 'ids array is NULL' in lib.mavd_last_error().decode(), (name, n)
            r.step([2, 0])                  # nothing ran: the streams are where they were
    # every non-stream Farneback call ends every stream: the step names the ended stream, then a restart works
    pair = torch.from_numpy(np.stack([r.cams.seqs[0][0]] * 2)).to(eng.device)
    samples, imu = r.samples[:1], _imu(1, 0)
    bgr_host = np.zeros((2, 240, 320), np.uint8)
    recs = np.empty((1,), dtype=np.dtype(_lib.FrameRecord))
    enders = [lambda: eng.farneback(pair, n_pairs=1, pair_stride=2),
              lambda: eng.process(pair, imu, samples, n_pairs=1, pair_stride=2),
              lambda: (eng.submit_host(0, bgr_host, imu, r.samples[:1].cpu().numpy(), n_pairs=1, pair_stride=2,
                                       records=recs), eng.wait_host(0))]
    for end in enders:
        end()
        for ids in ([0], [2, 0]):
            with pytest.raises(ValueError, match='stream %d is not started' % ids[0]):
                eng.stream_farneback(frames[:len(ids)], ids)
        r.start([2, 0])
        r.step([0, 2])
    # mavd_set_tuning keeps them
    eng.set_tuning(use_pdl=0)
    r.step([2, 0])
    r.close()


# ------------------------------------------------------------------------------------------------
# 4. graphs
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_changing_ids_replay_one_graph_and_match_direct_launches():
    """The ids are uploaded outside the captured sequence: steps with the same buffers and any ids replay one graph."""
    import torch
    from mav_detection_b200 import engine
    W, H, p = 640, 480, engine.SAMPLE_PARAMS
    eng, ref = engine.Engine(W, H, p, max_pairs=4), engine.Engine(W, H, p, max_pairs=4)
    cams = Cameras(W, H, 4, 20, seed=11)
    frames = torch.empty((2, H, W), dtype=torch.uint8, device=eng.device)
    flow = torch.empty((2, H, W, 2), device=eng.device)
    kept = [cams.next(s) for s in range(4)]
    for s in range(0, 4, 2):
        frames.copy_(torch.from_numpy(np.stack(kept[s:s + 2])))
        eng.stream_start(frames, [s, s + 1])
    schedule = [[0, 1], [2, 3], [1, 0], [3, 2], [0, 3], [1, 2], [2, 0], [3, 1]]
    for k, ids in enumerate(schedule * 2):
        if k == len(schedule):
            gs = eng.graph_stats()
            assert gs == {'captured': 2, 'direct': 0}, gs        # one for the starts, one for every step
            # the same schedule launched kernel by kernel, without programmatic dependent launch: bit-identical
            eng.set_tuning(use_graph=0, use_pdl=0)
        new = [cams.next(s) for s in ids]
        frames.copy_(torch.from_numpy(np.stack(new)))
        flow.fill_(float('nan'))
        eng.stream_farneback(frames, ids, out=flow)
        pairs = torch.from_numpy(np.stack([f for s, n in zip(ids, new) for f in (kept[s], n)])).to(ref.device)
        assert torch.equal(flow, ref.farneback(pairs, n_pairs=2, pair_stride=2)), (k, ids)
        for s, n in zip(ids, new):
            kept[s] = n
    eng.close()
    ref.close()


# ------------------------------------------------------------------------------------------------
# 5. host path
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('bgr', [False, True], ids=['gray', 'bgr'])
def test_host_submits_equal_the_device_stream_path(bgr):
    import torch
    from mav_detection_b200 import _lib, engine, sharded
    W, H, n = 640, 480, 3
    p = engine.SAMPLE_PARAMS
    host, dev = engine.Engine(W, H, p, max_pairs=n), engine.Engine(W, H, p, max_pairs=n)
    cams = Cameras(W, H, n, 8, seed=21)
    rng = np.random.default_rng(5)
    tint = lambda g: np.clip(g[..., None].astype(np.int16) + rng.integers(-9, 9, g.shape + (3,)), 0, 255).astype(np.uint8)
    first = [cams.next(s) for s in range(n)]
    first_bgr = [tint(f) for f in first]
    host.stream_start(host.bgr2gray(torch.from_numpy(np.stack(first_bgr)).cuda()) if bgr
                      else torch.from_numpy(np.stack(first)).cuda(), [0, 1, 2])
    dev.stream_start(dev.bgr2gray(torch.from_numpy(np.stack(first_bgr)).cuda()) if bgr
                     else torch.from_numpy(np.stack(first)).cuda(), [0, 1, 2])
    seg_all = (np.random.default_rng(9).random((n, H, W)) > 0.7).astype(np.uint8) * 255
    schedule = [[0, 1, 2], [2, 1], [1, 0, 2], [0], [2, 0], [1, 2, 0]]
    inflight = {}
    pb = host.packed_mask_bytes
    for k, ids in enumerate(schedule):
        slot = k % _lib.HOST_SLOTS
        if slot in inflight:
            host.wait_host(slot)
            _check_host(inflight.pop(slot))
        m = len(ids)
        new = [cams.next(s) for s in ids]
        frames = np.stack([tint(f) for f in new]) if bgr else np.stack(new)
        imu = _imu(m, k)
        samples = sharded.draw_all_samples(m, H, W, seed=k)
        seg = np.ascontiguousarray(seg_all[ids])
        seg_bits = host.pack_mask_host(seg)
        recs = np.empty((m,), dtype=engine.RECORD_DTYPE)
        fixed_bits = np.zeros((m, pb), np.uint8)
        flow = np.zeros((m, H, W, 2), np.float32)
        det = np.zeros((m, MAX_DET), dtype=engine.DETECTION_DTYPE)
        host.stream_submit_host(slot, frames, ids, imu, samples, seg=seg_bits, seg_packed=True, flow_out=flow,
                                fixed_out=fixed_bits, fixed_packed=True, records=recs, detections=det)
        # the device stream path on the same frames (gray as the copy-in stream converts them)
        d_frames = torch.from_numpy(frames).cuda()
        if bgr:
            d_frames = dev.bgr2gray(d_frames)
        out = _process_outputs(dev, m)
        d_rec, d_det = dev.stream_process(d_frames, ids, imu, torch.from_numpy(samples).cuda(),
                                          seg=torch.from_numpy(seg).cuda(), detections=MAX_DET, **out)
        inflight[slot] = (host, (recs, fixed_bits, flow, det),
                          (engine.Engine.records_to_numpy(d_rec), out['fixed_out'].cpu().numpy(),
                           out['flow_out'].cpu().numpy(), engine.Engine.detections_to_numpy(d_det)), (k, ids))
    for slot in list(inflight):
        host.wait_host(slot)
        _check_host(inflight.pop(slot))
    host.close()
    dev.close()


def _check_host(entry):
    from mav_detection_b200 import sharded
    eng, (recs, fixed_bits, flow, det), (d_rec, d_fixed, d_flow, d_det), where = entry
    assert not sharded.compare_records(recs, d_rec), where
    assert np.array_equal(eng.unpack_mask_host(fixed_bits), d_fixed), where
    assert np.array_equal(flow, d_flow), where
    for name in ('label', 'box', 'area', 'sum_x', 'sum_y'):
        assert np.array_equal(det[name], d_det[name]), (where, name)
    assert np.allclose(det['flow_sum'], d_det['flow_sum'], rtol=1e-12, atol=1e-9), where


# ------------------------------------------------------------------------------------------------
# 6. Farneback.process() on a stream of the shared engine
# ------------------------------------------------------------------------------------------------
class FakeCapture:
    def __init__(self, frames_bgr):
        self.frames, self.i = frames_bgr, 0

    def read(self):
        f = self.frames[min(self.i, len(self.frames) - 1)]
        self.i += 1
        return True, f.copy()


@pytest.mark.gpu
def test_farneback_process_with_other_users_of_the_shared_engine():
    """Two Farneback objects on the shared engine (one stream: the second pairs its frames explicitly, which ends the
    first one's stream) and a direct eng.farneback call interleave with a longer capture.  Every flow equals the explicit
    pair on a separate engine, and every image is the visualisation of that flow.  The first object pairs explicitly
    once its stream was ended before two calls in a row (t = 9 to 13), and goes back to its stream after a
    call with nobody else in between."""
    cv2 = pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine
    from mav_detection_b200.farneback import PROCESS_PARAMS, Farneback
    from oracle import vis_np
    W, H, T = 352, 240, 15         # a shared engine of its own (test_gpu_api.py's process() test uses 320 x 240)
    seqs = [_frames(W, H, T, 60), _frames(W, H, T, 61)]
    rng = np.random.default_rng(12)
    bgrs = [np.clip(s[..., None].astype(np.int16) + rng.integers(0, 40, (T, H, W, 3)) - 20, 0, 255).astype(np.uint8)
            for s in seqs]
    a = Farneback(FakeCapture(list(bgrs[0])), None)
    eng = a._eng
    assert a._stream == 0 and eng.max_pairs == 1
    b = Farneback(FakeCapture(list(bgrs[1])), None)
    assert b._eng is eng and b._stream is None
    ref = engine.Engine(W, H, PROCESS_PARAMS, max_pairs=1)
    p = PROCESS_PARAMS
    direct = torch.from_numpy(np.stack([seqs[0][0], seqs[1][0]])).to(eng.device)
    others, ended_in_a_row, paths = False, 0, []
    for t in range(1, T):
        users = [(a, 0)] if t in (3, 6, 13) else [(a, 0), (b, 1)]
        for fb, k in users:
            epoch = eng.stream_epoch
            out = fb.process()
            if fb is a:
                ended_in_a_row = ended_in_a_row + 1 if others else 0
                paths.append(eng.stream_epoch - epoch)          # 1: an explicit pair call, 0: a stream step
                assert paths[-1] == (ended_in_a_row >= 2), (t, ended_in_a_row)
                others = False
            else:
                others = True
            i = fb.capture.i - 1
            g0 = cv2.cvtColor(bgrs[k][i - 1], cv2.COLOR_BGR2GRAY)
            g1 = cv2.cvtColor(bgrs[k][i], cv2.COLOR_BGR2GRAY)
            want = ref.farneback(torch.from_numpy(np.stack([g0, g1])).to(ref.device), n_pairs=1)[0]
            assert torch.equal(fb.flow, want), (t, k)
            flow = fb.flow.cpu().numpy()
            mine, invalid = vis_np.process_visualisation(flow)
            assert not invalid and np.array_equal(out, mine), (t, k)
            cvf = cv2.calcOpticalFlowFarneback(g0, g1, None, p['pyr_scale'], p['levels'], p['winsize'],
                                               p['iterations'], p['poly_n'], p['poly_sigma'], p['flags'])
            assert np.linalg.norm(flow - cvf, axis=-1).mean() < EPE_MEAN_TOL, (t, k)
            ref_img, _ = vis_np.process_visualisation_cv2(cvf, (H, W, 3))
            assert (out == ref_img).all(-1).mean() > 0.99, (t, k)
        if t % 4 == 0:
            eng.farneback(direct, n_pairs=1)          # a direct call by another user of the engine
            others = True
    assert 0 < sum(paths) < len(paths) and paths[-1] == 0, paths     # both paths taken; back on the stream at the end
    ref.close()
