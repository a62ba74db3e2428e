"""Cost of the per-frame detection tables (mavd_process_det) on bench.py's 1920x1080 workloads.

For C2, c2rot and c2dense it times one 64-pair step of the device path (resident frames, graph replay, CUDA events)
without a table and with max_det 32 and 256, the three arms alternating step by step so that clock drift and other
tenants hit them alike, and prints the added milliseconds per step.  It also reports how often the largest detection
of a frame is the synthetic MAV: the frame's segmentation box contains the detection's centroid.

    python tools/detections_cost.py [--steps 20] [--workloads c2,c2rot,c2dense] [--out result.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card() -> dict:
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=20).stdout.strip()
        name, power, clock = [p.strip() for p in out.split(',')]
        return {'gpu': name, 'power_limit': power, 'sm_max_clock': clock}
    except Exception as e:      # the numbers still stand, without the card's settings beside them
        return {'gpu': 'unknown (%s)' % e}


def run(name: str, steps: int) -> dict:
    import torch
    import bench
    from mav_detection_b200 import _lib, engine
    wl = bench.build_workload(name)
    W, H, B, params, seq = wl['W'], wl['H'], wl['B'], wl['params'], wl['seq']
    nb = bench.N_BATCHES
    eng = engine.Engine(W, H, params, max_pairs=B)
    frames = torch.from_numpy(seq.frames).cuda()
    seg = torch.from_numpy(seq.segmentation).cuda()
    samples = torch.from_numpy(wl['samples']).cuda()
    fixed = torch.empty((B, H, W), dtype=torch.uint8, device='cuda')
    records = torch.empty((B, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
    det = {md: torch.empty((B, md, engine.DETECTION_DTYPE.itemsize), dtype=torch.uint8, device='cuda')
           for md in (32, 256)}
    imus = [engine.make_imu(B, seq.omega[b * B + 1:b * B + 1 + B], seq.dt,
                            derotate=[(b * B + i) >= 1 for i in range(B)]) for b in range(nb)]
    stream = torch.cuda.Stream()

    def step(s: int, md: int) -> None:
        b = s % nb
        f0 = b * B
        aux = eng._aux(None, seg[f0 + 1:f0 + B + 1], None, B)
        _lib.check(eng.lib.mavd_process_det(eng._h, frames[f0:f0 + B + 1].data_ptr(), B, 1, imus[b],
                                            C.byref(eng.detect_params), samples[f0:f0 + B].data_ptr(), C.byref(aux),
                                            None, None, fixed.data_ptr(), records.data_ptr(), md,
                                            det[md].data_ptr() if md else None, eng._stream()))

    arms = (0, 32, 256)
    times = {md: [] for md in arms}
    largest_is_mav = []
    with torch.cuda.stream(stream):
        for s in range(nb):
            for md in arms:
                step(s, md)                              # capture every (batch, arm) launch sequence
        torch.cuda.synchronize()
        for s in range(steps):
            for md in (arms if s % 2 == 0 else arms[::-1]):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step(s, md)
                e1.record()
                e1.synchronize()
                times[md].append(e0.elapsed_time(e1))
                if md == 32 and s < nb:
                    rec = eng.records_to_numpy(records)
                    tab = det[32].cpu().numpy().view(engine.DETECTION_DTYPE)[..., 0]
                    for f in range(B):
                        d = tab[f, 0]
                        x0, y0, x1, y1 = (int(v) for v in rec[f]['stats']['seg_bbox'])
                        if d['label'] == 0 or x0 < 0:
                            largest_is_mav.append(False)
                            continue
                        cx, cy = d['sum_x'] / d['area'], d['sum_y'] / d['area']
                        largest_is_mav.append(bool(x0 <= cx <= x1 and y0 <= cy <= y1))
    gs = eng.graph_stats()
    eng.close()
    med = {md: float(np.median(times[md])) for md in arms}
    return {'workload': name, 'pairs_per_step': B, 'steps': steps, 'graphs': gs,
            'ms_per_step': {('none' if md == 0 else 'max_det_%d' % md): round(med[md], 4) for md in arms},
            'added_ms_per_step': {'max_det_%d' % md: round(med[md] - med[0], 4) for md in (32, 256)},
            'spread_ms_none': [round(float(np.min(times[0])), 4), round(float(np.max(times[0])), 4)],
            'largest_detection_is_mav': '%d / %d frames' % (sum(largest_is_mav), len(largest_is_mav))}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--workloads', default='c2,c2rot,c2dense')
    ap.add_argument('--out', default=None, help='also write the result as JSON to this path')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('detections_cost.py measures on the GPU: no CUDA device')
    res = {'card': card(), 'results': [run(w, args.steps) for w in args.workloads.split(',')]}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
