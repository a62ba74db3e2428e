#!/usr/bin/env python
"""Benchmark of the mav-detection hot path (Farneback flow -> derotate -> FoE -> phi/masks -> components).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload c2|c2rot|c2dense|c2gauss|c2w21|c2ref|c1|c3|c4|all] [--tune field=value,...]
                    [--dump-outputs DIR]

One "step" = one pass of the whole hot path over one batch of frame pairs taken from a synthetic
sequence that is resident in HBM (device arm) / in pinned host memory (e2e).  Prints ONE JSON line.
Metric: BASELINE.json -> 1080p frame-pairs/sec (flow+FoE+mask), plus % of HBM roofline of the fused
Farneback iteration kernel.  `--impl reference` times the reference's own CPU path (cv2's Farneback +
the NumPy restatement of the reference's FoE/phi/mask code in oracle/) on the host cores.
`--workload all` measures C2 (the headline) and adds one line per other configuration under `extra`.
`--dump-outputs DIR` writes what the headline workload's last timed step returned to its caller as DIR/<name>.npy
(see dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

JSON_OUT = sys.stdout     # main() swaps this for a private handle on the real stdout

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SAMPLE = dict(pyr_scale=0.5, levels=5, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2, flags=0)
REFPRM = dict(pyr_scale=0.4, levels=1, winsize=12, iterations=10, poly_n=8, poly_sigma=1.2, flags=0)
WORKLOADS = {
    # name: (W, H, farneback params, pairs per step, label, sequence options)
    'c2': (1920, 1080, SAMPLE, 64,
           'C2: synthetic AirSim-like 1920x1080 sequence, Farneback (0.5,5,15,3,5,1.2,0) 6 pyramid images', {}),
    'c2rot': (1920, 1080, SAMPLE, 64,
              'C2 with IMU rotation omega=(0.002,-0.001,0.0005) rad/frame (derotation not a no-op)',
              dict(with_rotation=True)),
    'c2dense': (1920, 1080, SAMPLE, 64,
                'C2 frames under a sideways translation: no FoE consensus, ~100 % of the pixels in both masks '
                '(dense residual / components stress)', dict(motion='translate')),
    'c2gauss': (1920, 1080, dict(SAMPLE, flags=256), 64,
                'C2 with OPTFLOW_FARNEBACK_GAUSSIAN (flags=256): Gaussian windows on the TMA-staged iteration kernel', {}),
    'c2w21': (1920, 1080, dict(SAMPLE, winsize=21), 64,
              'C2 with winsize 21 (half-width 10, outside the TMA kernel\'s 5..8): the generic iteration kernel', {}),
    'c2ref': (1920, 1080, REFPRM, 32, "C2': 1920x1080 with the reference's own parameters (0.4,1,12,10,8,1.2,0)", {}),
    'c1': (640, 480, REFPRM, 1, 'C1: one 640x480 pair, reference parameters', {}),
    'c3': (640, 480, SAMPLE, 64, 'C3: 640x480, 64 pairs per launch', {}),
    'c4': (3840, 2160, dict(SAMPLE, levels=7, iterations=10), 8,
           'C4: 3840x2160, 7 pyramid images, winsize 15, 10 iterations', {}),
}
EXTRA_ORDER = ['c2rot', 'c2dense', 'c2ref', 'c1', 'c3', 'c4']
N_BATCHES = 4          # distinct resident batches cycled through (working set per step >> L2 anyway)
DUMP_MASK_SAMPLES = 1 << 21   # fixed-mask pixels kept by --dump-outputs (C2's 64 masks hold 133 M pixels)
DUMP_SEED = 0


def hbm_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 25 ms from before the warm-up on; stop(t0, t1) reports the
    samples that arrived inside the timed region [t0, t1] (host clock), or, if the region was too short to catch two
    of them, all samples taken while the GPU was busy (the warm-up steps run the same kernels back to back)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap,utilization.gpu')

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '25'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float = 0.0, t1: float = float('inf')):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = []
        for ts, ln in self.lines:
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 8:
                continue
            try:
                rows.append((ts, float(parts[0]), float(parts[1]), float(parts[2]),
                             [n for n, v in zip(names, parts[3:7]) if v.lower().startswith('active')], float(parts[7])))
            except ValueError:
                continue
        timed = [r for r in rows if t0 <= r[0] <= t1 + 0.03]
        window = 'timed region'
        if len(timed) < 2:
            timed = [r for r in rows if r[5] >= 50.0 or r[3] >= 300.0] or rows
            window = 'warm-up + timed region (GPU busy)'
        sm = [r[1] for r in timed]
        reasons = sorted({n for r in timed for n in r[4]})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max((r[2] for r in rows), default=None),
                'power_w_max': max((r[3] for r in timed), default=None), 'samples': len(timed), 'window': window,
                'reasons': reasons}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def build_workload(name: str, rank: int = 0, pairs: int = 0):
    from mav_detection_b200 import synth
    W, H, params, B, label, opts = WORKLOADS[name]
    B = pairs or B
    n_frames = N_BATCHES * B + 1
    seq = synth.make_sequence(W, H, n_frames, seq=rank, **opts)
    rs = np.random.RandomState(1000 + rank)   # legacy generator = the stream np.random.randint draws from
    samples = np.empty((N_BATCHES * B, 4000), np.int32)
    for i in range(N_BATCHES * B):
        samples[i, :2000] = rs.randint(0, H, 2000)
        samples[i, 2000:] = rs.randint(0, W, 2000)
    return dict(name=name, W=W, H=H, params=params, B=B, label=label, seq=seq, samples=samples)


def dump_outputs(out_dir: str, records: np.ndarray, fixed: np.ndarray) -> None:
    """Writes one step's outputs, as a caller of Engine.process receives them, to out_dir/<name>.npy: each field of
    the per-pair records as float64 (records_<field>, records_stats_<field>), and the (pairs, H, W) fixed masks as
    float32, whole (fixed) when they hold at most DUMP_MASK_SAMPLES pixels, else as a seeded sample of them
    (fixed_sample, taken at the flat indices stored as float64 in fixed_sample_index)."""
    out = {}
    for name in records.dtype.names:
        if name == 'stats':
            for sub in records.dtype['stats'].names:
                out['records_stats_' + sub] = np.asarray(records['stats'][sub], np.float64)
        else:
            out['records_' + name] = np.asarray(records[name], np.float64)
    flat = fixed.reshape(-1)
    if flat.size <= DUMP_MASK_SAMPLES:
        out['fixed'] = np.asarray(fixed, np.float32)
    else:
        idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, flat.size, DUMP_MASK_SAMPLES))
        out['fixed_sample_index'] = idx.astype(np.float64)
        out['fixed_sample'] = flat[idx].astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def level_sizes(W, H, params):
    """Pyramid image sizes, finest first (SURVEY §8 a2)."""
    k, s = 0, 1.0
    while k < params['levels']:
        s *= params['pyr_scale']
        if W * s < 32 or H * s < 32:
            break
        k += 1
    out = []
    for li in range(k + 1):
        sc = params['pyr_scale'] ** li
        out.append((int(np.rint(W * sc)), int(np.rint(H * sc))))
    return out


def algorithmic_bytes(W, H, params, B, n_frames):
    """SURVEY §8(d) stage-graph compulsory bytes per launch group of each profiled kernel class, for B pairs."""
    lv = level_sizes(W, H, params)
    px = [w * h for w, h in lv]
    n0, it = px[0], params['iterations']
    return {
        'pyramid': n_frames * sum(n0 + 4 * p for p in px[1:]) if len(px) > 1 else 0,
        'polyexp': n_frames * (n0 * (1 + 20) + sum(24 * p for p in px[1:])),
        'matrices': B * (sum(68 * p for p in px[:-1]) + 60 * px[-1] + sum(8 * p for p in px[1:])),
        'iter_full': B * 88.0 * n0 * max(it - 1, 0),
        'iter_full_last': B * 28.0 * n0,
        'iter_coarse': B * sum((88.0 * (it - 1) + 28.0) * p for p in px[1:]),
        'residual': B * 12.0 * n0,          # flow 8 + sky/seg 2 -> two masks 2
        'ccl': B * 5.0 * n0,
    }


def survey_bytes_per_pair(W, H, params):
    """SURVEY §8(d) stage-graph compulsory HBM bytes of one INDEPENDENT pair (both frames' pyramid and expansion counted
    for every pair; 992.4 MB for C2): the denominator of the whole-path roofline figure quoted since round 1."""
    px = [w * h for w, h in level_sizes(W, H, params)]
    n0, sp, it = px[0], sum(px), params['iterations']
    pyramid = 2 * sum(n0 + 4 * p for p in px)
    polyexp = 2 * 24 * sp
    flow_init = 8 * px[-1] + sum(8 * px[l + 1] + 8 * px[l] for l in range(len(px) - 1))
    matrices = 68 * sp
    iters = (88 * (it - 1) + 28) * sp
    post = 16 * n0
    return pyramid + polyexp + flow_init + matrices + iters + post


def cpu_one_pair(args):
    """The reference's CPU path for one pair: cv2 Farneback + restated derotate/FoE/phi/masks."""
    import cv2
    from oracle import detect_np as dn
    prev, nxt, params, omega, dt, ry, rx, idx = args
    t0 = time.perf_counter()
    flow = cv2.calcOpticalFlowFarneback(prev, nxt, None, params['pyr_scale'], params['levels'], params['winsize'],
                                        params['iterations'], params['poly_n'], params['poly_sigma'], params['flags'])
    t1 = time.perf_counter()
    sky = np.zeros(prev.shape, bool)
    dn.frame_pipeline(idx, flow, omega, dt, sky, ry, rx)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def _cpu_init():
    import cv2
    cv2.setNumThreads(1)   # one pair per core: OpenCV's Farneback core is single-threaded anyway


class CpuReference:
    """The reference's CPU path on a pool of host processes (one frame pair per process at a time)."""

    def __init__(self, wl, workers: int):
        import multiprocessing as mp
        self.wl, self.workers = wl, workers
        self.pool = mp.get_context('spawn').Pool(workers, initializer=_cpu_init)

    def jobs(self, n_pairs: int):
        seq, wl = self.wl['seq'], self.wl
        out = []
        for i in range(n_pairs):
            p = i % (seq.frames.shape[0] - 1)
            out.append((seq.frames[p], seq.frames[p + 1], wl['params'], seq.omega[p + 1], seq.dt,
                        wl['samples'][p, :2000], wl['samples'][p, 2000:], 1 + p))
        return out

    def step(self, n_pairs: int):
        """Returns (pairs/s, mean flow ms, mean post ms, seconds)."""
        jobs = self.jobs(n_pairs)
        t0 = time.perf_counter()
        res = self.pool.map(cpu_one_pair, jobs, chunksize=1)
        dt = time.perf_counter() - t0
        return (n_pairs / dt, 1e3 * float(np.mean([r[0] for r in res])), 1e3 * float(np.mean([r[1] for r in res])), dt)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_workers() -> int:
    return max(1, min(os.cpu_count() or 1, 32))


def metric_name(W):
    return '1080p frame-pairs/sec (flow+FoE+mask)' if W == 1920 else 'frame-pairs/sec (flow+FoE+mask)'


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import cv2
    wl = build_workload('c2' if args.workload == 'all' else args.workload, 0, args.pairs)
    workers = cpu_workers()
    per_step = workers
    ref = CpuReference(wl, workers)
    vals = []
    for s in range(args.warmup + args.steps):
        r = ref.step(per_step)
        if s >= args.warmup:
            vals.append(r)
    ref.close()
    v = float(np.sum([per_step for _ in vals]) / np.sum([x[3] for x in vals]))
    line = {
        'impl': 'reference',
        'metric': metric_name(wl['W']),
        'value': v, 'unit': 'pairs/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * float(np.mean([x[3] for x in vals])), 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl['label'], 'pairs_per_step': per_step},
        'cpu_baseline': {'value': v, 'unit': 'pairs/s', 'cores': workers, 'kind': 'port',
                         'sample': '%d pairs/step on %d processes (cv2.calcOpticalFlowFarneback %s, the library the '
                                   'reference calls, + oracle/detect_np restatement of derotate/FoE/phi/masks); per '
                                   'pair: flow %.0f ms, post %.0f ms; host has %d logical CPUs'
                                   % (per_step, workers, cv2.__version__, float(np.mean([x[1] for x in vals])),
                                      float(np.mean([x[2] for x in vals])), os.cpu_count() or 0)},
        'e2e': {'value': v, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), file=JSON_OUT, flush=True)


# ------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------
def measure(name, args, steps, world, rank, local, headline):
    """One workload on this rank's GPU.  Returns the fields of the JSON line (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from mav_detection_b200 import engine
    from mav_detection_b200._lib import HOST_SLOTS

    wl = build_workload(name, rank, args.pairs)
    W, H, B, params = wl['W'], wl['H'], wl['B'], wl['params']
    seq = wl['seq']
    eng = engine.Engine(W, H, params, max_pairs=B, device=local)
    if args.tune:
        eng.set_tuning(**engine.parse_tuning(args.tune))
    dev = torch.device('cuda', local)
    stream = torch.cuda.Stream(device=dev)

    # resident inputs (device arm) and pinned host inputs (e2e arm)
    frames_d = torch.from_numpy(seq.frames).to(dev)
    seg_d = torch.from_numpy(seq.segmentation).to(dev)
    samples_d = torch.from_numpy(wl['samples']).to(dev)
    fixed_d = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
    records_d = torch.empty((B, engine.RECORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    gathered = [torch.empty_like(records_d) for _ in range(world)] if world > 1 else None
    imus = []
    for b in range(N_BATCHES):
        first = b * B
        imus.append(engine.make_imu(B, seq.omega[first + 1:first + 1 + B], seq.dt,
                                    derotate=[(first + i) >= 1 for i in range(B)]))
    side = torch.cuda.Stream(device=dev) if world > 1 else None

    def step(s):
        b = s % N_BATCHES
        f0 = b * B
        eng.process(frames_d[f0:f0 + B + 1], imus[b], samples_d[f0:f0 + B], seg=seg_d[f0 + 1:f0 + B + 1],
                    fixed_out=fixed_d, records=records_d)
        if world > 1:
            # only detection boxes / FoE points cross NVLink: one small all_gather per batch, side stream
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                dist.all_gather(gathered, records_d)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    warm = max(args.warmup, N_BATCHES + 1)     # every resident batch once: its launch sequence is captured then
    sampler = ClockSampler(local)
    if rank == 0 and headline:
        sampler.start()
    with torch.cuda.stream(stream):
        for s in range(warm):
            step(s)
        sync_all()
        # (1) the timed region: K steps as the caller sees them (graph replay when tuning.use_graph)
        launches0 = eng.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        t_host0 = time.time()
        e0.record()
        for s in range(steps):
            step(warm + s)
        if world > 1:
            torch.cuda.current_stream(dev).wait_stream(side)
        e1.record()
        sync_all()
        t_host1 = time.time()
        elapsed_ms = e0.elapsed_time(e1)
        clocks = sampler.stop(t_host0, t_host1) if (rank == 0 and headline) else None
        launches = eng.launch_count() - launches0
        if args.dump_outputs and headline and rank == 0:
            # the last timed step's outputs, before the passes below overwrite them
            dump_outputs(args.dump_outputs, eng.records_to_numpy(records_d), fixed_d.cpu().numpy())
        # (2) per-kernel-class device times: the same steps again with CUDA events around every launch group
        # (profiling launches kernel by kernel, so it is kept out of the timed region above)
        psteps = max(2, min(steps, 8))
        if args.device_only:
            psteps, prof = 1, {}
        else:
            eng.profile_enable(True)
            for s in range(psteps):
                step(warm + s)
            sync_all()
            prof = eng.profile_read()
            eng.profile_enable(False)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    value = world * B * steps / (elapsed_ms * 1e-3)

    if args.device_only:
        line = None
        if rank == 0:
            line = {'metric': metric_name(W), 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': steps,
                    'warmup': warm, 'ms_per_step': elapsed_ms / steps, 'gpu_launches': int(launches),
                    'config': {'workload': wl['label'], 'pairs_per_step': B, 'device_only': True}}
        eng.close()
        return line

    # ---- e2e: host buffers through the C-ABI host call, copies inside the timed region ----
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
        t.numpy()[...] = a
        return t.numpy()
    npx = W * H
    pb = eng.packed_mask_bytes
    frames_h = pinned(seq.frames)
    seg_h = pinned(seq.segmentation)
    segbits_h = pinned(eng.pack_mask_host(seq.segmentation))
    samples_h = pinned(wl['samples'])
    fixed_h = [pinned(np.zeros((B, H, W), np.uint8)) for _ in range(HOST_SLOTS)]
    fixedbits_h = [pinned(np.zeros((B, pb), np.uint8)) for _ in range(HOST_SLOTS)]
    rec_h = [pinned(np.zeros((B,), engine.RECORD_DTYPE).view(np.uint8)).view(engine.RECORD_DTYPE)
             for _ in range(HOST_SLOTS)]

    def host_pass(packed: bool, copy_only: bool, n_steps: int) -> float:
        """pairs/s of this rank's pipelined host calls: batch s's host->device copies overlap batch s-1's kernels
        and batch s-2's device->host copies (mavd_submit_host_ex / mavd_wait_host, HOST_SLOTS staging sets)."""
        def one(s):
            b = s % N_BATCHES
            f0 = b * B
            slot = s % HOST_SLOTS
            eng.wait_host(slot)
            if packed:
                eng.submit_host(slot, frames_h[f0:f0 + B + 1], imus[b], samples_h[f0:f0 + B],
                                seg=segbits_h[f0 + 1:f0 + B + 1], fixed_out=fixedbits_h[slot], records=rec_h[slot],
                                seg_packed=True, fixed_packed=True, copy_only=copy_only)
            else:
                eng.submit_host(slot, frames_h[f0:f0 + B + 1], imus[b], samples_h[f0:f0 + B],
                                seg=seg_h[f0 + 1:f0 + B + 1], fixed_out=fixed_h[slot], records=rec_h[slot],
                                copy_only=copy_only)

        def drain():
            for slot in range(HOST_SLOTS):
                eng.wait_host(slot)
        with torch.cuda.stream(stream):
            # warm-up: every (staging slot, resident batch) combination once, so that each launch sequence the timed
            # steps replay has been captured (and every lazily allocated staging buffer exists)
            n_warm = HOST_SLOTS * N_BATCHES if not copy_only else 3
            for s in range(n_warm):
                one(s)
            drain()
            sync_all()
            t0 = time.perf_counter()
            for s in range(n_steps):
                one(n_warm + s)
            drain()                       # every step's records and masks have landed in host memory
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return world * B * n_steps / dt

    e2e_value = host_pass(True, False, steps)
    h2d = (B + 1) * npx + B * pb + B * 4000 * 4
    d2h = B * engine.RECORD_DTYPE.itemsize + B * pb
    e2e_detail = None
    if headline:
        short = max(4, steps // 2)
        e2e_detail = {
            'packed_masks': e2e_value,
            'byte_masks': host_pass(False, False, short),
            'copy_only_packed_masks': host_pass(True, True, short),
            'copy_only_byte_masks': host_pass(False, True, short),
            'bytes_per_step_byte_masks': {'h2d': int((B + 1) * npx + B * npx + B * 16000),
                                          'd2h': int(B * engine.RECORD_DTYPE.itemsize + B * npx)},
            'note': 'copy_only_* = the same host calls with the compute skipped (MAVD_HOST_COPY_ONLY): the host-feed '
                    'ceiling of this box at this N; byte_masks = segmentation in / estimate_fixed out as uint8 images',
        }

    line = None
    if rank == 0:
        peak, peak_src = hbm_peak()
        alg = algorithmic_bytes(W, H, params, B, B + 1)
        per_class = {}
        for k, (ms, n) in prof.items():
            if n <= 0:
                continue
            ms_step = ms / psteps
            ent = {'ms_per_step': round(ms_step, 4)}
            if alg.get(k) and k not in ('pyramid', 'polyexp'):      # those two overlap the side stream: wall time, not kernel time
                ent['algorithmic_gb_per_step'] = round(alg[k] / 1e9, 3)
                ent['frac_of_hbm_peak'] = round(alg[k] / (ms_step * 1e-3) / 1e9 / peak, 3)
            per_class[k] = ent
        it_ms, it_n = prof['iter_full']
        roof = None
        if it_n > 0:
            dur_s = it_ms * 1e-3 / it_n
            ab = 88.0 * W * H * B
            achieved = ab / dur_s / 1e9
            traffic, traffic_src = None, None
            try:
                with open(os.path.join(ROOT, 'profiles', 'iter_kernel_traffic.json')) as f:
                    tj = json.load(f)
                per_pair = tj.get(name + '_per_pair') or (tj.get('c2_per_pair') if name.startswith('c2') and
                                                          params == SAMPLE else None)
                traffic = per_pair * B if per_pair else None      # bytes per launch, like `achieved`
                traffic_src = tj.get('source')
            except Exception:
                pass
            roof = {'bound': 'hbm', 'kernel': 'iter_box_tma_kernel<m, not-last> (fused Farneback iteration), finest level',
                    'achieved': achieved, 'peak': peak, 'peak_source': peak_src, 'unit': 'GB/s', 'frac': achieved / peak,
                    'traffic': traffic, 'traffic_source': traffic_src,
                    'frac_by_traffic': (traffic / dur_s / 1e9 / peak) if traffic else None,
                    'us_per_launch': dur_s * 1e6, 'us_per_pair': dur_s * 1e6 / B,
                    'algorithmic_bytes_per_launch': ab, 'launches_timed': it_n}
        cpu = None
        if world == 1 and headline and not args.no_cpu:
            workers = cpu_workers()
            ref = CpuReference(wl, workers)
            ref.step(workers)                                  # warm-up: page in cv2, first touch
            v, flow_ms, post_ms, dt = ref.step(2 * workers if workers <= 8 else workers)
            ref.close()
            import cv2
            cpu = {'value': v, 'unit': 'pairs/s', 'cores': workers, 'kind': 'port',
                   'sample': '%d processes, one pair of this workload at a time (cv2 %s Farneback + oracle/detect_np); '
                             'per pair: flow %.0f ms, FoE/phi/masks %.0f ms; host has %d logical CPUs'
                             % (workers, cv2.__version__, flow_ms, post_ms, os.cpu_count() or 0)}
        whole_alg = sum(alg.values())
        whole_survey = survey_bytes_per_pair(W, H, params) * B
        line = {
            'metric': metric_name(W),
            'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': steps, 'warmup': warm,
            'ms_per_step': elapsed_ms / steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': wl['label'], 'pairs_per_step': B, 'frames_resident': int(seq.frames.shape[0]),
                       'l2_policy': 'inputs larger than L2: each step streams a %.1f GB working set'
                                    % (eng.workspace_bytes / 1e9),
                       'sharding': 'each rank runs its own sequence; records all_gathered over NCCL per step'
                                   if world > 1 else 'single GPU',
                       'tuning': eng.get_tuning(), 'launch_sequences': eng.graph_stats()},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': 'pairs/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'call': 'mavd_submit_host_ex/mavd_wait_host (C ABI, pinned host buffers, %d batches in flight; '
                            'segmentation in and estimate_fixed out at 1 bit per pixel)' % HOST_SLOTS},
            'e2e_detail': e2e_detail,
            'gpu_launches': int(launches),
            'roofline': roof,
            'whole_path_frac_of_hbm_peak': round(whole_survey / (elapsed_ms / steps * 1e-3) / 1e9 / peak, 3),
            'whole_path_bytes': {'survey_8d_independent_pairs_mb_per_pair': round(whole_survey / B / 1e6, 1),
                                 'sequence_mode_shared_frames_mb_per_pair': round(whole_alg / B / 1e6, 1),
                                 'frac_sequence_mode': round(whole_alg / (elapsed_ms / steps * 1e-3) / 1e9 / peak, 3)},
            'kernel_classes': per_class,
            'cpu_baseline': cpu,
        }
    eng.close()
    del frames_d, seg_d, samples_d, fixed_d, records_d
    torch.cuda.empty_cache()
    return line


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    parity = None
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        # multi-GPU parity before any timing: a sharded sequence must reproduce the single-GPU records
        from mav_detection_b200 import sharded
        ok, parity = sharded.parity_check(local)
        if not ok:
            if rank == 0:
                print('bench.py: ' + parity, file=sys.stderr, flush=True)
            dist.destroy_process_group()
            sys.exit(3)
    main_name = 'c2' if args.workload == 'all' else args.workload
    line = measure(main_name, args, args.steps, world, rank, local, True)
    if rank == 0 and parity:
        line['config']['sharded_parity'] = parity
    if args.workload == 'all':
        extra = {}
        for name in EXTRA_ORDER:
            steps = max(4, min(args.steps, 20 if WORKLOADS[name][0] <= 1920 else 6))
            if name == 'c1':
                steps = max(steps, 200)
            sub = measure(name, args, steps, world, rank, local, False)
            if rank == 0:
                extra[name] = {k: sub[k] for k in ('value', 'unit', 'ms_per_step', 'steps', 'e2e', 'gpu_launches', 'roofline',
                                                   'whole_path_frac_of_hbm_peak', 'kernel_classes')}
                extra[name]['workload'] = sub['config']['workload']
                extra[name]['pairs_per_step'] = sub['config']['pairs_per_step']
        if rank == 0:
            line['extra'] = extra
    if rank == 0:
        print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS) + ['all'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--device-only', action='store_true',
                    help='warm-up + timed device steps only (no per-kernel event pass, no e2e, no CPU leg): the command '
                         'ncu captures, so that its launch list is whole steps of the hot path and nothing else')
    ap.add_argument('--pairs', type=int, default=0, help='frame pairs per step (default: the workload\'s)')
    ap.add_argument('--tune', default=os.environ.get('MAVD_TUNE', ''),
                    help='mavd_tuning fields, e.g. pair_group=8,use_graph=0 (A/B runs; results never depend on them)')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='write the outputs of the last timed step of the headline workload (rank 0) to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    # stdout carries the JSON line and nothing else: keep a private handle on the real stdout for it and point file
    # descriptor 1 at stderr, so that whatever a library prints (NCCL's version banner, worker processes) lands there
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
