"""Cost of the sparse feature path on 1920x1080 synthetic frames (the flagship frame size).

Times, with CUDA events on resident frames, good_features(2000, 0.01, 7, blockSize 7) on 65 frames and pyr_lk (21 x 21,
maxLevel 3, default criteria) on the 64 pairs those frames make, fed by the corners.  Both arms run warm-ups first and
then alternate step by step.  Prints the card's name and power limit beside the numbers, and cv2's time for the same
work on this host (one frame and one pair, scaled to the batch).

    python tools/sparse_cost.py [--steps 10] [--out result.json]
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


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import cv2
    import torch
    from mav_detection_b200 import engine, synth
    W, H, P = 1920, 1080, 64
    seq = synth.make_sequence(W, H, P + 1, seq=0, with_rotation=True)
    frames = torch.from_numpy(np.ascontiguousarray(seq.frames)).cuda()
    eng = engine.Engine(W, H, max_pairs=P)
    corners, counts = eng.good_features(frames, 2000, 0.01, 7, 7)
    times = {'good_features_65': [], 'pyr_lk_64': []}
    arms = {'good_features_65': lambda: eng.good_features(frames, 2000, 0.01, 7, 7),
            'pyr_lk_64': lambda: eng.pyr_lk(frames, corners[:P], n_points=counts[:P], pair_stride=1)}
    for fn in arms.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    for _ in range(args.steps):
        for name, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b))
    a0, b0 = seq.frames[0], seq.frames[1]
    t = time.perf_counter()
    p = cv2.goodFeaturesToTrack(a0, 2000, 0.01, 7, blockSize=7)
    t_g = time.perf_counter() - t
    t = time.perf_counter()
    cv2.calcOpticalFlowPyrLK(a0, b0, p, None, winSize=(21, 21), maxLevel=3)
    t_l = time.perf_counter() - t
    res = dict(card(), steps=args.steps, mean_corners=float(counts.float().clamp(max=2000).mean()),
               cv2_threads=cv2.getNumThreads())
    for name, v in times.items():
        res[name + '_ms_median'] = float(np.median(v))
        res[name + '_ms_min'] = float(np.min(v))
    res['cv2_good_features_65_ms'] = t_g * 1e3 * (P + 1)
    res['cv2_pyr_lk_64_ms'] = t_l * 1e3 * P
    print(json.dumps(res))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == '__main__':
    main()
