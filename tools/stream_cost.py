"""What frame streams save: each new frame is expanded once instead of being re-sent and re-expanded with its pair.

(a) 64 cameras at 1920x1080 with OpenCV's sample parameters (bench.py's C2): one step = one new frame per camera.
    stream   mavd_stream_process on the 64 new frames (each camera's previous frame is kept on the device)
    pairs    mavd_process with pair_stride 2 on the same 64 (previous, new) pairs: 128 frames
    Both device-resident (frames already in HBM) and through the host-submit path (pinned host frames, three slots in
    flight: the stream arm moves 64 frames per step, the pair arm 128).  Each arm has its own handle; the arms alternate
    round by round after warm-ups, in reversed order every other round.  Times are host clocks around `steps` steps that end in a device synchronise.
    Camera c's frame at time t is frame c + t of one sequence.  Every stream round first restarts the streams with time
    0 (outside the timed window), and its step k takes time k + 1: both arms time exactly the same (k, k + 1) pairs.
(b) Farneback.process() at 640x480 with the reference's parameters, per call (gray conversion, flow, visualisation,
    copy of the image to the host): on a stream of its engine, and with every stream of the engine taken, which is the
    explicit pair call it made before streams existed.  Then two Farneback objects that alternate on one engine with a
    single stream (the second one pairs explicitly, which ends the first one's stream every frame), against the same
    two on an engine whose stream is taken (both pair explicitly); per pair of calls.

Prints one JSON object: per arm the median and the spread (min, max) over the rounds, the card's name and power limit.

    python tools/stream_cost.py [--rounds 7] [--steps 10] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.detections_cost import card  # noqa: E402

def _order(arms: dict, r: int) -> list:
    """The arms of round r: in the given order on even rounds, reversed on odd ones, so that no arm always runs first."""
    items = list(arms.items())
    return items if r % 2 == 0 else items[::-1]


def _stat(v):
    return {'median': float(np.median(v)), 'min': float(np.min(v)), 'max': float(np.max(v))}


def cameras_64(rounds: int, steps: int) -> dict:
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, P = 1920, 1080, 64
    seq = synth.make_sequence(W, H, P + steps, seq=0)
    # step k: the new frames are time k + 1, the pairs (time k, time k + 1); all resident
    new = [np.ascontiguousarray(seq.frames[k + 1:k + 1 + P]) for k in range(steps)]
    pairs = [np.ascontiguousarray(np.stack([seq.frames[k:k + P], seq.frames[k + 1:k + 1 + P]], 1).reshape(2 * P, H, W))
             for k in range(steps)]
    ids = list(range(P))
    imu = engine.make_imu(P, ang=np.tile([0.002, -0.001, 0.0005], (P, 1)), dt=0.05)
    samples_h = sharded.draw_all_samples(P, H, W, seed=0)
    samples = torch.from_numpy(samples_h).cuda()
    es, ep = engine.Engine(W, H, engine.SAMPLE_PARAMS, P), engine.Engine(W, H, engine.SAMPLE_PARAMS, P)
    new_d = [torch.from_numpy(a).cuda() for a in new]
    pairs_d = [torch.from_numpy(a).cuda() for a in pairs]
    rec_s = torch.empty((P, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    rec_p = torch.empty_like(rec_s)

    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = a
        return t.numpy()
    new_h, pairs_h = [pinned(a) for a in new], [pinned(a) for a in pairs]
    recs_h = [np.empty((P,), dtype=engine.RECORD_DTYPE) for _ in range(3)]

    time0 = torch.from_numpy(np.ascontiguousarray(seq.frames[:P])).cuda()
    arms = {
        'stream_device': lambda k: es.stream_process(new_d[k], ids, imu, samples, records=rec_s),
        'pairs_device': lambda k: ep.process(pairs_d[k], imu, samples, n_pairs=P, pair_stride=2, records=rec_p),
    }

    def host_arm(eng, stream):
        def run(k):
            slot = k % 3
            eng.wait_host(slot)
            if stream:
                eng.stream_submit_host(slot, new_h[k], ids, imu, samples_h, records=recs_h[slot])
            else:
                eng.submit_host(slot, pairs_h[k], imu, samples_h, n_pairs=P, pair_stride=2, records=recs_h[slot])
        return run
    arms['stream_host'] = host_arm(es, True)
    arms['pairs_host'] = host_arm(ep, False)

    def drain():
        for e in (es, ep):
            for slot in range(3):
                e.wait_host(slot)
        torch.cuda.synchronize()

    def prepare(name):
        drain()
        if name.startswith('stream'):
            es.stream_start(time0, ids)     # the streams keep time 0 again
            torch.cuda.synchronize()

    for name, fn in arms.items():       # warm-up: every graph of the timed rounds is captured here
        prepare(name)
        for k in range(steps):
            fn(k)
    times = {name: [] for name in arms}
    for r in range(rounds):
        for name, fn in _order(arms, r):
            prepare(name)
            t0 = time.perf_counter()
            for k in range(steps):
                fn(k)
            drain()
            times[name].append((time.perf_counter() - t0) * 1e3 / steps)
    es.close()
    ep.close()
    out = {'workload': '64 cameras, 1920x1080, Farneback (0.5,5,15,3,5,1.2,0), one new frame per camera per step',
           'steps_per_round': steps, 'rounds': rounds}
    for name, v in times.items():
        out[name + '_ms_per_step'] = _stat(v)
        out[name + '_new_frames_per_s'] = float(P * 1e3 / np.median(v))
    for where in ('device', 'host'):
        out['stream_gain_' + where] = float(np.median(times['pairs_' + where]) / np.median(times['stream_' + where]) - 1)
    return out


class _Capture:
    def __init__(self, frames):
        self.frames, self.i = frames, 0

    def read(self):
        f = self.frames[self.i % len(self.frames)]
        self.i += 1
        return True, f


def farneback_process(rounds: int, calls: int) -> dict:
    import torch
    from mav_detection_b200 import engine, synth
    from mav_detection_b200.farneback import PROCESS_PARAMS, Farneback
    W, H = 640, 480
    seq = synth.make_sequence(W, H, 16, seq=1)
    rng = np.random.default_rng(0)
    bgr = [np.clip(f[..., None].astype(np.int16) + rng.integers(-10, 10, (H, W, 3)), 0, 255).astype(np.uint8)
           for f in seq.frames]
    with_stream = Farneback(_Capture(bgr), None, engine=engine.Engine(W, H, PROCESS_PARAMS, 1))
    taken = engine.Engine(W, H, PROCESS_PARAMS, 1)
    taken.open_stream()                       # no free stream: the explicit pair call
    pairs = Farneback(_Capture(bgr), None, engine=taken)
    assert with_stream._stream is not None and pairs._stream is None
    shared = engine.Engine(W, H, PROCESS_PARAMS, 1)
    two_shared = [Farneback(_Capture(bgr), None, engine=shared), Farneback(_Capture(bgr[::-1]), None, engine=shared)]
    taken2 = engine.Engine(W, H, PROCESS_PARAMS, 1)
    taken2.open_stream()
    two_taken = [Farneback(_Capture(bgr), None, engine=taken2), Farneback(_Capture(bgr[::-1]), None, engine=taken2)]
    arms = {'process_stream': [with_stream], 'process_pairs': [pairs],
            'two_users_one_stream': two_shared, 'two_users_no_stream': two_taken}
    for fbs in arms.values():
        for _ in range(10):
            for fb in fbs:
                fb.process()
    torch.cuda.synchronize()
    times = {name: [] for name in arms}
    for r in range(rounds):
        for name, fbs in _order(arms, r):
            t0 = time.perf_counter()
            for _ in range(calls):
                for fb in fbs:
                    fb.process()          # ends in the device-to-host copy of the image
            times[name].append((time.perf_counter() - t0) * 1e3 / calls)
    out = {'workload': 'Farneback.process(), 640x480 BGR, reference parameters (0.4,1,12,10,8,1.2,0)',
           'calls_per_round': calls, 'rounds': rounds}
    for name, v in times.items():
        out[name + '_ms_per_call'] = _stat(v)
    out['stream_gain'] = float(np.median(times['process_pairs']) / np.median(times['process_stream']) - 1)
    out['two_users_gain'] = float(np.median(times['two_users_no_stream']) / np.median(times['two_users_one_stream']) - 1)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--calls', type=int, default=200)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not 1 <= args.steps <= 12:
        # one resident batch per step: with the start and the three host slots a handle then holds up to 16 captured
        # launch sequences, its cache size; more would recapture every step
        ap.error('--steps must be in 1..12')
    res = dict(card())
    res['cameras_64'] = cameras_64(args.rounds, args.steps)
    res['farneback_process'] = farneback_process(args.rounds, args.calls)
    print(json.dumps(res))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
