"""GPU: whole-path parity at the BASELINE sizes (1080p C2, one 4K pair, the dense-mask case), the 1-bit-per-pixel wire
format, the batched ground-truth-flow reduction, graph replay vs direct launches, and several engines / devices in
one process.  Everything goes through the C ABI (mav_detection_b200.engine is a ctypes shim)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _samples(n, H, W, seed):
    from oracle import detect_np as dn
    np.random.seed(seed)
    return np.stack([np.concatenate(dn.draw_sample_indices(H, W)) for _ in range(n)]).astype(np.int32)


def _check_against_chained_oracle(seq, params, flow, fixed, rec, samples, first_index=0, cv2_pairs=()):
    """records / masks of every pair against the oracle chained on OUR flow (bit-exact stages), boxes against the
    labelling oracle, and the flow itself against cv2 for the pairs listed in cv2_pairs."""
    import cv2
    from oracle import ccl_np
    from oracle import detect_np as dn
    n = flow.shape[0]
    for p in range(n):
        if p in cv2_pairs:
            ref = cv2.calcOpticalFlowFarneback(seq.frames[p], seq.frames[p + 1], None, params['pyr_scale'],
                                               params['levels'], params['winsize'], params['iterations'],
                                               params['poly_n'], params['poly_sigma'], params['flags'])
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


def _run_device(eng, seq, n, samples, first_index=0):
    import torch
    from mav_detection_b200 import engine
    H, W = seq.frames.shape[1:]
    imu = engine.make_imu(n, seq.omega[1:n + 1], seq.dt, derotate=[(first_index + i) >= 1 for i in range(n)])
    flow_t = torch.empty((n, H, W, 2), dtype=torch.float32, device=eng.device)
    fixed_t = torch.empty((n, H, W), dtype=torch.uint8, device=eng.device)
    rec = eng.process(torch.from_numpy(seq.frames[:n + 1]).to(eng.device), imu, torch.from_numpy(samples).to(eng.device),
                      seg=torch.from_numpy(seq.segmentation[1:n + 1].copy()).to(eng.device), flow_out=flow_t,
                      fixed_out=fixed_t)
    return flow_t.cpu().numpy(), fixed_t.cpu().numpy(), eng.records_to_numpy(rec)


@pytest.mark.parametrize('rot', [False, True])
def test_whole_path_1080p_c2(rot):
    """BASELINE configs[1] geometry: 1920x1080, Farneback (0.5,5,15,3,5,1.2,0); with and without IMU rotation."""
    pytest.importorskip('cv2')
    from mav_detection_b200 import engine, synth
    W, H, n = 1920, 1080, 3
    seq = synth.make_sequence(W, H, n + 1, seq=11, with_rotation=rot)
    params = dict(engine.SAMPLE_PARAMS)
    samples = _samples(n, H, W, 31)
    eng = engine.Engine(W, H, params, max_pairs=n)
    flow, fixed, rec = _run_device(eng, seq, n, samples)
    _check_against_chained_oracle(seq, params, flow, fixed, rec, samples, cv2_pairs=(0, 2))
    eng.close()


def test_whole_path_4k_pair():
    """BASELINE configs[3] geometry: one 3840x2160 pair, 7 pyramid images, winsize 15, 10 iterations."""
    pytest.importorskip('cv2')
    from mav_detection_b200 import engine, synth
    W, H = 3840, 2160
    seq = synth.make_sequence(W, H, 2, seq=12, with_rotation=True)
    params = dict(pyr_scale=0.5, levels=7, winsize=15, iterations=10, poly_n=5, poly_sigma=1.2, flags=0)
    samples = _samples(1, H, W, 32)
    eng = engine.Engine(W, H, params, max_pairs=1)
    assert len(eng.levels) == 7
    flow, fixed, rec = _run_device(eng, seq, 1, samples, first_index=1)
    _check_against_chained_oracle(seq, params, flow, fixed, rec, samples, first_index=1, cv2_pairs=(0,))
    eng.close()


def test_whole_path_dense_masks():
    """Sideways translation: the flow lines are parallel, there is no FoE consensus ((0, 0)), and nearly every pixel
    ends up in both masks — one image-sized component for the labelling, every word on the statistics path."""
    pytest.importorskip('cv2')
    from mav_detection_b200 import engine, synth
    W, H, n = 640, 480, 3
    seq = synth.make_sequence(W, H, n + 1, seq=13, motion='translate')
    params = dict(engine.SAMPLE_PARAMS)
    samples = _samples(n, H, W, 33)
    eng = engine.Engine(W, H, params, max_pairs=n)
    flow, fixed, rec = _run_device(eng, seq, n, samples)
    assert fixed.mean() > 0.3                         # the case is what it claims to be: large connected masks
    _check_against_chained_oracle(seq, params, flow, fixed, rec, samples, cv2_pairs=(1,))
    eng.close()


@pytest.mark.parametrize('size', [(64, 48), (203, 131), (1920, 1080)])
def test_pack_unpack_mask_kernels(size):
    import torch
    from mav_detection_b200 import engine
    W, H = size
    rng = np.random.default_rng(4)
    mask = (rng.random((3, H, W)) < 0.3).astype(np.uint8) * rng.integers(1, 256, (3, H, W)).astype(np.uint8)
    mask[2] = 0
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=1)
    pb = eng.packed_mask_bytes
    assert pb % 4 == 0 and pb * 8 >= W * H
    bits = eng.pack_mask(torch.from_numpy(mask).cuda()).cpu().numpy()
    ref = eng.pack_mask_host(mask)
    assert bits.shape == (3, pb) and np.array_equal(bits, ref)
    flat = np.packbits(mask.reshape(3, -1) != 0, axis=-1, bitorder='little')
    assert np.array_equal(bits[:, :flat.shape[1]], flat) and not bits[:, flat.shape[1]:].any()
    for value in (1, 255):
        back = eng.unpack_mask(torch.from_numpy(bits).cuda(), value).cpu().numpy()
        assert np.array_equal(back, (mask != 0).astype(np.uint8) * value)
    assert np.array_equal(eng.unpack_mask_host(bits), (mask != 0).astype(np.uint8))
    eng.close()


def test_host_path_packed_masks_equal_byte_masks():
    """mavd_submit_host with MAVD_HOST_SEG_PACKED | MAVD_HOST_SKY_PACKED | MAVD_HOST_FIXED_PACKED returns the same
    records and (after unpacking) the same estimate_fixed masks as the byte-mask call; copy-only skips the compute."""
    from mav_detection_b200 import engine, synth
    W, H, n = 320, 240, 4
    seq = synth.make_sequence(W, H, n + 1, seq=14, with_rotation=True)
    samples = _samples(n, H, W, 34)
    imu = engine.make_imu(n, seq.omega[1:], seq.dt, derotate=[i >= 1 for i in range(n)])
    sky = np.zeros((H, W), np.uint8)
    sky[:30] = 1                                              # a sky band: both masks are forced to zero there
    seg = np.ascontiguousarray(seq.segmentation[1:])
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    fixed_a = np.zeros((n, H, W), np.uint8)
    rec_a = eng.process_host(seq.frames, imu, samples, sky=sky, seg=seg, fixed_out=fixed_a).copy()
    fixed_bits = np.zeros((n, eng.packed_mask_bytes), np.uint8)
    rec_b = eng.process_host(seq.frames, imu, samples, sky=eng.pack_mask_host(sky), seg=eng.pack_mask_host(seg),
                             fixed_out=fixed_bits, sky_packed=True, seg_packed=True, fixed_packed=True).copy()
    from mav_detection_b200 import sharded
    assert sharded.compare_records(rec_b, rec_a) == []
    assert np.array_equal(eng.unpack_mask_host(fixed_bits), fixed_a)
    assert not fixed_a[:, :30].any() and fixed_a.any()
    assert (rec_a['stats']['positives'] == (seg > 127).reshape(n, -1).sum(1)).all()
    # copy-only: the bytes move, nothing is computed (the outputs are whatever the staging held)
    before = eng.launch_count()
    eng.wait_host(1)
    eng.submit_host(1, seq.frames, imu, samples, seg=eng.pack_mask_host(seg), fixed_out=fixed_bits, seg_packed=True,
                    fixed_packed=True, copy_only=True)
    eng.wait_host(1)
    assert eng.launch_count() - before == 2               # unpack + pack
    # out-of-range sample indices are rejected on the host path
    bad = samples.copy()
    bad[1, 5] = H
    with pytest.raises(ValueError):
        eng.process_host(seq.frames, imu, bad)
    eng.close()


def test_out_of_range_samples_are_clamped_on_the_device_path():
    """A stale sample table (wrong resolution) must not read outside the flow field: indices are clamped in the
    kernel, the result equals the oracle fed the clamped indices."""
    import torch
    from mav_detection_b200 import engine
    from oracle import detect_np as dn
    W, H = 160, 120
    rng = np.random.default_rng(6)
    ys, xs = np.mgrid[0:H, 0:W]
    flow = (np.stack([(xs - 70.5) * 0.05, (ys - 50.5) * 0.05], -1) + rng.normal(0, 0.05, (H, W, 2))).astype(np.float32)
    smp = _samples(1, 4 * H, 4 * W, 35)                         # drawn for a 4x larger frame
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=1)
    imu = engine.make_imu(1, derotate=[False])
    foe, cnt = eng.foe(torch.from_numpy(flow[None]).cuda(), imu, torch.from_numpy(smp).cuda())
    ry, rx = np.minimum(smp[0, :2000], H - 1), np.minimum(smp[0, 2000:], W - 1)
    assert tuple(foe.cpu().numpy()[0]) == dn.foe_dense(flow, ry, rx)
    with pytest.raises(ValueError):
        eng.detect(torch.from_numpy(flow[None]).cuda(), imu, torch.from_numpy(smp.astype(np.int64)).cuda())
    with pytest.raises(ValueError):
        eng.detect(torch.from_numpy(flow[None]).cuda(), imu, torch.from_numpy(smp))          # CPU tensor
    eng.close()


@pytest.mark.parametrize('host', [False, True])
def test_ground_truth_flow_sum_in_the_batch(host):
    """mavd_aux_inputs.gt_flow: Detector.derotate(gt_flow) summed over segmentation > 127, per frame, in the same
    device call (processor.py:309-310,344) — float32 pass-through for frame 0, float64 after derotation otherwise."""
    import torch
    from mav_detection_b200 import engine, synth
    from oracle import detect_np as dn
    W, H, n = 320, 240, 3
    seq = synth.make_sequence(W, H, n + 1, seq=15, with_rotation=True)
    rng = np.random.default_rng(16)
    gt = rng.normal(0, 2, (n, H, W, 2)).astype(np.float32)
    flow = rng.normal(0, 2, (n, H, W, 2)).astype(np.float32)
    samples = _samples(n, H, W, 36)
    imu = engine.make_imu(n, seq.omega[1:], seq.dt, derotate=[i >= 1 for i in range(n)])
    seg = np.ascontiguousarray(seq.segmentation[1:])
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    if host:
        rec = eng.detect_host(flow, imu, samples, seg=seg, gt_flow=gt)
    else:
        rec = eng.records_to_numpy(eng.detect(torch.from_numpy(flow).cuda(), imu, torch.from_numpy(samples).cuda(),
                                              seg=torch.from_numpy(seg).cuda(), gt_flow=torch.from_numpy(gt).cuda()))
    for i in range(n):
        gd = dn.derotate(i, gt[i], seq.omega[i + 1], seq.dt)
        fd = dn.derotate(i, flow[i], seq.omega[i + 1], seq.dt)
        m = seg[i] > 127
        assert m.sum() > 0
        assert np.allclose(rec[i]['stats']['gt_flow_sum'], gd[m].astype(np.float64).sum(axis=0), rtol=1e-10, atol=1e-9)
        assert np.allclose(rec[i]['stats']['seg_flow_sum'], fd[m].astype(np.float64).sum(axis=0), rtol=1e-10, atol=1e-9)
    # without a ground-truth flow the sum stays zero
    rec0 = eng.detect_host(flow, imu, samples, seg=seg)
    assert not rec0['stats']['gt_flow_sum'].any()
    eng.close()


def test_processor_batches_the_ground_truth_flow():
    """Processor.run_detection on a dataset WITH ground-truth flow (the reference's SimData case): drone_flow_pixels is
    the derotated ground-truth average (processor.py:344,359) and the batch stays one device call."""
    import logging
    from mav_detection_b200 import engine, synth
    from mav_detection_b200.processor import Processor
    from mav_detection_b200.run_config import RunConfig
    from oracle import detect_np as dn
    W, H, F = 320, 240, 7
    seq = synth.make_sequence(W, H, F, seq=17, with_rotation=True)
    rng = np.random.default_rng(18)
    flows = rng.normal(0, 2, (F - 1, H, W, 2)).astype(np.float32)
    gts = rng.normal(0, 2, (F - 1, H, W, 2)).astype(np.float32)
    ds = synth.SyntheticDataset(seq, flows=flows, gt_flows=gts)
    RunConfig.register_dataset(RunConfig.DatasetType.SIMULATION, lambda logger, sequence: ds)
    cfg = RunConfig(logging.getLogger('test'), 'simulation', 'synthetic', False, False, False, True, False, False,
                    'FLOW_FOE_CLUSTERING')
    proc = Processor(cfg, flow_source='dataset', batch_frames=4, farneback_params=engine.SAMPLE_PARAMS,
                     write_results=False)
    calls = []
    orig = proc.engine.detect_host
    proc.engine.detect_host = lambda *a, **k: (calls.append(1), orig(*a, **k))[1]
    launches = proc.engine.launch_count()
    res = proc.run_detection()
    assert len(calls) == 2                                      # 6 frames in batches of 4: two device calls in all
    assert sorted(res) == list(range(F - 1))
    for i in range(F - 1):
        gd = dn.derotate(i, gts[i], seq.omega[i], seq.dt)
        avg = gd[seq.segmentation[i] > 127].astype(np.float64).mean(axis=0)
        assert np.allclose(res[i].drone_flow_pixels, avg, rtol=1e-9, atol=1e-12), i
    assert proc.engine.launch_count() - launches < 80          # not one residual launch per frame
    proc.release()


def test_graph_replay_equals_direct_launches_across_tunings():
    """tuning.use_graph: the captured launch sequence (side stream included) replays the same kernels with the same
    arguments — flows, masks and records are bit-equal to the kernel-by-kernel path, on a user stream and on the
    legacy default stream, first call (capture) and later calls (replay), and after a tuning change."""
    import torch
    from mav_detection_b200 import engine, sharded, synth
    W, H, n = 640, 480, 4
    seq = synth.make_sequence(W, H, n + 1, seq=19, with_rotation=True)
    samples = _samples(n, H, W, 37)
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    assert eng.get_tuning()['use_graph'] == 1
    eng.set_tuning(use_graph=0)
    flow0, fixed0, rec0 = _run_device(eng, seq, n, samples)
    direct_launches = eng.launch_count()
    eng.set_tuning(use_graph=1)
    for trial in range(3):                                      # capture, replay, replay
        before = eng.launch_count()
        flow1, fixed1, rec1 = _run_device(eng, seq, n, samples)
        assert np.array_equal(flow1, flow0) and np.array_equal(fixed1, fixed0), trial
        assert sharded.compare_records(rec1, rec0) == [], trial
    with torch.cuda.stream(torch.cuda.Stream()):
        flow2, fixed2, rec2 = _run_device(eng, seq, n, samples)
        torch.cuda.current_stream().synchronize()
    assert np.array_equal(flow2, flow0) and np.array_equal(fixed2, fixed0)
    # buffers differ from call to call in _run_device (fresh tensors): each is its own graph; the launch counter counts
    # the replayed kernels too
    assert eng.launch_count() - before > 20
    # every sequence was captured and instantiated (programmatic dependent launches included): nothing fell back
    assert eng.get_tuning()['use_pdl'] == 1
    gs = eng.graph_stats()
    assert gs['captured'] >= 1 and gs['direct'] == 0, gs
    eng.set_tuning(iter_small_tiles=0, polyexp_tma=0, pyr_staged=0)    # other launch shapes, same results
    flow3, fixed3, rec3 = _run_device(eng, seq, n, samples)
    assert np.array_equal(flow3, flow0) and np.array_equal(fixed3, fixed0)
    assert direct_launches > 20
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize('graph', [0, 1])
def test_programmatic_dependent_launch_changes_nothing(graph):
    """tuning.use_pdl: kernels made resident behind their predecessor (griddepcontrol) wait for its completion before
    they touch memory — flows, masks and records are bit-equal to the fully serialised launches, kernel by kernel and
    inside captured graphs, over repeated calls (a kernel released too early would read a half-written field)."""
    from mav_detection_b200 import engine, sharded, synth
    W, H, n = 640, 480, 6
    seq = synth.make_sequence(W, H, n + 1, seq=23, with_rotation=True)
    samples = _samples(n, H, W, 41)
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    eng.set_tuning(use_pdl=0, use_graph=graph)
    flow0, fixed0, rec0 = _run_device(eng, seq, n, samples)
    eng.set_tuning(use_pdl=1, use_graph=graph)
    for trial in range(4):
        flow1, fixed1, rec1 = _run_device(eng, seq, n, samples)
        assert np.array_equal(flow1, flow0) and np.array_equal(fixed1, fixed0), trial
        assert sharded.compare_records(rec1, rec0) == [], trial
    if graph:
        gs = eng.graph_stats()
        assert gs['captured'] >= 1 and gs['direct'] == 0, gs
    eng.close()


def test_two_engines_in_one_process():
    """Two handles side by side (different geometry, same device), used alternately; on a box with two GPUs the second
    one lives on cuda:1 while cuda:0 stays the current device (per-device kernel attributes, device guard)."""
    import torch
    from mav_detection_b200 import engine, synth
    dev1 = 1 if torch.cuda.device_count() > 1 else 0
    p = dict(engine.SAMPLE_PARAMS)        # winsize 15: the 73 KB dynamic-shared-memory iteration kernel
    a = engine.Engine(320, 240, p, max_pairs=1, device=0)
    b = engine.Engine(352, 288, p, max_pairs=1, device=dev1)
    sa, sb = synth.make_sequence(320, 240, 2, seq=20), synth.make_sequence(352, 288, 2, seq=21)
    cur = torch.cuda.current_device()
    for _ in range(2):
        fa = a.farneback(torch.from_numpy(sa.frames).to(a.device))
        fb = b.farneback(torch.from_numpy(sb.frames).to(b.device))
        assert torch.cuda.current_device() == cur           # the calls restore the caller's device
    torch.cuda.synchronize(a.device)
    torch.cuda.synchronize(b.device)
    from oracle import farneback_np as fbn
    for f, s in ((fa, sa), (fb, sb)):
        ref = fbn.calc_optical_flow_farneback(s.frames[0], s.frames[1], None, **p)
        assert np.linalg.norm(f[0].cpu().numpy() - ref, axis=-1).mean() < 1e-3
    g = b.bgr2gray(torch.zeros((4, 4, 3), dtype=torch.uint8, device=b.device))
    assert g.device == b.device
    a.close()
    b.close()


def test_vis_kernels_match_the_reference_outputs(golden_dir):
    """mavd_phi_colormap / mavd_mask_overlay through the reference-named im_helpers functions, against the golden vectors
    the reference's own im_helpers / processor.py statements produced (tests/golden/make_golden_vis_flo.py)."""
    import os
    from mav_detection_b200 import im_helpers
    from oracle import vis_np
    g = np.load(os.path.join(golden_dir, 'vis_ref.npz'))
    for name, phi in (('f64', g['phi64']), ('f32', g['phi32'])):
        rgb = im_helpers.to_rgb(phi, max_value=180.0)
        assert np.array_equal(rgb, g['phi_rgb_' + name]), name
        assert np.array_equal(im_helpers.apply_colormap(rgb), g['phi_jet_' + name]), name
        assert np.array_equal(im_helpers.apply_colormap(rgb, max_value=180.0), g['phi_jet_max_' + name]), name
        assert np.array_equal(im_helpers.apply_colormap(phi, max_value=180.0)[1:], g['phi_jet_' + name][1:]), name
    vis, mask_rgb = im_helpers.mask_overlay(g['frame'], g['fixed'], want_mask_rgb=True)
    assert np.array_equal(vis, g['mask_vis']) and np.array_equal(mask_rgb, g['result_img'])
    gray = g['frame'][..., 1].copy()
    assert np.array_equal(im_helpers.mask_overlay(gray, g['fixed']), vis_np.mask_overlay(gray, g['fixed'])[0])
    # every byte value through the overlay, masked and unmasked
    v = np.arange(256, dtype=np.uint8).reshape(16, 16)
    frame = np.stack([v, v[::-1], v.T], -1).copy()
    for fixed in (np.zeros((16, 16), bool), np.ones((16, 16), bool)):
        assert np.array_equal(im_helpers.mask_overlay(frame, fixed), vis_np.mask_overlay(frame, fixed)[0])
    # a 1080p phi field straight from the residual stage (float64) and its colour image
    rng = np.random.default_rng(7)
    big = rng.uniform(0, 180, (1080, 1920))
    assert np.array_equal(im_helpers.apply_colormap(im_helpers.to_rgb(big, 180.0)),
                          vis_np.apply_colormap_jet(vis_np.to_rgb(big, 180.0)))


def test_flo_cache_round_trip_through_the_processor(tmp_path):
    """flow_source='farneback' with a FloCache writes <index:06d>.flo per frame in the reference's layout; a second
    Processor with flow_source='dataset' over CachedFlowDataset (the Dataset.get_flow_uv seam) reproduces every
    FrameResult of the first run."""
    import logging
    import torch
    from mav_detection_b200 import engine, flow_cache, synth, utils
    from mav_detection_b200.processor import Processor
    from mav_detection_b200.run_config import RunConfig
    W, H, F = 320, 240, 8
    params = dict(engine.SAMPLE_PARAMS)
    seq = synth.make_sequence(W, H, F, seq=22, with_rotation=True)
    cache = flow_cache.FloCache(str(tmp_path / 'output' / 'inference' / 'run.epoch-0-flow-field'))

    def run(ds, source, fc):
        RunConfig.register_dataset(RunConfig.DatasetType.SIMULATION, lambda logger, sequence: ds)
        cfg = RunConfig(logging.getLogger('test'), 'simulation', 'synthetic', False, False, False, True, False, False,
                        'FLOW_FOE_CLUSTERING')
        np.random.seed(5)
        proc = Processor(cfg, flow_source=source, batch_frames=3, farneback_params=params, write_results=False,
                         flow_cache=fc)
        res = proc.run_detection()
        eng = proc.engine
        proc.release()
        return res, eng
    first, eng = run(synth.SyntheticDataset(seq), 'farneback', cache)
    cache.flush()
    assert sorted(os.listdir(cache.directory)) == ['%06d.flo' % i for i in range(F - 1)]
    fr = torch.from_numpy(seq.frames).to(eng.device)
    flows = np.concatenate([eng.farneback(fr[b:b + 4]).cpu().numpy() for b in range(0, F - 1, 3)])    # max_pairs is 3
    for i in range(F - 1):
        assert np.array_equal(utils.read_flow(flow_cache.flo_path(cache.directory, i)), flows[i]), i
    # device batches go through the pinned double buffer
    cache2 = flow_cache.FloCache(str(tmp_path / 'again'))
    dev = torch.from_numpy(flows).to(eng.device)
    cache2.put_batch(0, dev[:4])
    cache2.put_batch(4, dev[4:])
    for i in range(F - 1):
        assert np.array_equal(cache2.get_flow_uv(i), flows[i]), i
    second, _ = run(flow_cache.CachedFlowDataset(synth.SyntheticDataset(seq), cache), 'dataset', None)
    assert sorted(second) == sorted(first)
    for i in first:
        a, b = first[i], second[i]
        assert a.foe_dense == b.foe_dense and (a.tpr, a.fpr, a.tpr_fixed, a.fpr_fixed) == (b.tpr, b.fpr, b.tpr_fixed, b.fpr_fixed)
        assert np.allclose(a.drone_flow_pixels, b.drone_flow_pixels, rtol=1e-12)


@pytest.mark.parametrize('size', [(1920, 1080), (640, 480), (203, 131), (64, 48), (100, 37)])
def test_ccl_dense_and_structured_masks(size):
    """The run-based labelling on everything from 100 % foreground to noise: one image-sized component, checkerboards
    (8-connected through diagonals only), stripes, 50 % noise (thousands of components, more than the 32 boxes kept),
    widths that are / are not multiples of 4 and of the 128-pixel unit (units straddling rows, several rows per unit)."""
    import torch
    from mav_detection_b200 import engine
    from oracle import ccl_np
    W, H = size
    rng = np.random.default_rng(W * 7 + H)
    ys, xs = np.mgrid[0:H, 0:W]
    masks = np.stack([
        np.ones((H, W), np.uint8),                                   # one component
        ((xs + ys) % 2).astype(np.uint8),                            # checkerboard
        (xs % 3 == 0).astype(np.uint8),                              # vertical stripes
        (ys % 2 == 0).astype(np.uint8) * (xs % 7 != 3),              # broken horizontal stripes
        (rng.random((H, W)) < 0.5).astype(np.uint8),                 # noise
        (rng.random((H, W)) < 0.93).astype(np.uint8),                # almost full
        ((xs // 5 + ys // 3) % 2).astype(np.uint8) * 200,            # blocks touching at corners, value != 1
        np.zeros((H, W), np.uint8),
    ]).astype(np.uint8)
    masks[7, H // 2, :] = 1
    masks[7, :, W // 3] = 1
    masks[7, 0, 0] = masks[7, H - 1, W - 1] = 1
    n = masks.shape[0]
    eng = engine.Engine(W, H, engine.SAMPLE_PARAMS, max_pairs=n)
    for want_labels in (True, False):
        labels, boxes, cnt = eng.ccl(torch.from_numpy(masks).cuda(), want_labels=want_labels)
        boxes, cnt = boxes.cpu().numpy(), cnt.cpu().numpy()
        for i in range(n):
            ref, stats = ccl_np.label(masks[i])
            assert cnt[i] == ref.max(), (i, cnt[i], ref.max())
            if want_labels:
                assert np.array_equal(labels[i].cpu().numpy(), ref), i
            k = min(32, stats.shape[0])
            assert np.array_equal(boxes[i, :k], stats[:k]), i
    eng.close()


@pytest.mark.parametrize('size', [(1920, 1080), (752, 480), (333, 257), (64, 48), (1024, 96)])
@pytest.mark.parametrize('poly_n', [5, 8, 3])
def test_tma_staged_polyexp_is_bit_identical(size, poly_n):
    """tuning.polyexp_tma: the expansion tile staged by one TMA box (u8 frame box + in-kernel 3x3 blur at level 0, float
    image box at the coarser levels) against the per-thread-load kernel: every R plane of every level bit-equal —
    interior tiles, all four borders (REFLECT_101 ring of the blur, replicated halo of the expansion), widths that
    are not multiples of the tile (and, for 333, not of 16: level 0 then falls back to the load kernel)."""
    import torch
    from mav_detection_b200 import engine, synth
    W, H = size
    s = synth.make_sequence(W, H, 2, seq=23)
    p = dict(pyr_scale=0.5, levels=3, winsize=15, iterations=1, poly_n=poly_n, poly_sigma=1.2, flags=0)
    eng = engine.Engine(W, H, p, max_pairs=1)
    frames = torch.from_numpy(s.frames).cuda()
    got = {}
    for tma in (1, 0):
        eng.set_tuning(polyexp_tma=tma)
        flow = eng.farneback(frames).cpu().numpy()
        got[tma] = [eng.tap('R', lvl, j).cpu().numpy() for lvl in range(len(eng.levels)) for j in (0, 1)] + [flow]
    for a, b in zip(got[1], got[0]):
        assert np.array_equal(a, b), float(np.abs(a - b).max())
    eng.close()


@pytest.mark.parametrize('winsize', [12, 15, 17])
def test_small_tile_iteration_is_bit_identical(winsize):
    """tuning.iter_small_tiles: launches too small to fill the GPU with 64 x 32 tiles (one 640x480 pair; the coarse
    levels) run the fused iteration on 64 x 16 tiles.  Same sums, same order: flows bit-equal, every level."""
    import torch
    from mav_detection_b200 import engine, synth
    W, H = 640, 480
    s = synth.make_sequence(W, H, 2, seq=24)
    p = dict(pyr_scale=0.5, levels=3, winsize=winsize, iterations=3, poly_n=5, poly_sigma=1.2, flags=0)
    eng = engine.Engine(W, H, p, max_pairs=1)
    frames = torch.from_numpy(s.frames).cuda()
    got = {}
    for small in (1, 0):
        eng.set_tuning(iter_small_tiles=small)
        flow = eng.farneback(frames).cpu().numpy()
        got[small] = [flow] + [eng.tap('flow', lvl, 0).cpu().numpy() for lvl in range(1, len(eng.levels))] + \
            [eng.tap('M', lvl, 0).cpu().numpy() for lvl in range(len(eng.levels))]
    for a, b in zip(got[1], got[0]):
        assert np.array_equal(a, b), float(np.abs(a - b).max())
    eng.force_generic_iteration(True)
    assert np.array_equal(eng.farneback(frames).cpu().numpy(), got[1][0])
    eng.close()


@pytest.mark.parametrize('winsize', [11, 13, 15, 17])
def test_gaussian_windows_on_the_tma_iteration_kernel(winsize):
    """OPTFLOW_FARNEBACK_GAUSSIAN with winsize/2 in 5..8 runs on the TMA-staged kernel (both tile heights) since round
    2: equal to the generic kernel (same filter expressions) and to cv2 within the flow tolerance."""
    cv2 = pytest.importorskip('cv2')
    import torch
    from mav_detection_b200 import engine, synth
    s = synth.make_sequence(700, 500, 3, seq=25)
    p = dict(pyr_scale=0.5, levels=3, winsize=winsize, iterations=3, poly_n=5, poly_sigma=1.2, flags=256)
    eng = engine.Engine(700, 500, p, max_pairs=2)
    frames = torch.from_numpy(s.frames).cuda()
    a = eng.farneback(frames).cpu().numpy()
    eng.force_generic_iteration(True)
    b = eng.farneback(frames).cpu().numpy()
    eng.force_generic_iteration(False)
    eng.set_tuning(iter_small_tiles=0)
    c = eng.farneback(frames).cpu().numpy()
    assert np.array_equal(a, c), float(np.abs(a - c).max())                    # 64 x 16 vs 64 x 32 tiles
    assert np.array_equal(a, b), float(np.abs(a - b).max())                    # TMA vs generic
    ref = cv2.calcOpticalFlowFarneback(s.frames[0], s.frames[1], None, 0.5, 3, winsize, 3, 5, 1.2, 256)
    epe = np.linalg.norm(a[0] - ref, axis=-1)
    assert epe.mean() < 1e-4 and epe.max() < 5e-3, (epe.mean(), epe.max())
    eng.close()


@pytest.mark.parametrize('size', [(1920, 1080), (640, 480), (648, 488), (3840, 2160), (2048, 1024), (644, 484),
                                  (640, 481), (640, 200, 0.498)])
def test_pyramid_sweep_equals_the_generic_kernels(size):
    """tuning.pyr_sweep: the exact power-of-two levels of a pyr_scale 0.5 pyramid computed by one sweep down the frame
    (vertical passes) and the vectorised horizontal pass equal the generic kernels' images bit for bit, for every band
    count, on noise frames (every REFLECT_101 border row / column matters); sizes whose coarse levels are not exact
    decimations (1080 / 16, 484 / 8) mix both kinds of kernels.  An odd height (481) leaves level 1 a horizontal
    decimation only: no sweep, level 1's horizontal pass on its own.  640 x 200 at pyr_scale 0.498 (levels 319 x 100,
    159 x 50) is the reverse: the sweep runs without level 1's horizontal pass."""
    import torch
    from mav_detection_b200 import engine
    W, H, pyr_scale = size if len(size) == 3 else size + (0.5,)
    p = dict(engine.SAMPLE_PARAMS)
    p['levels'] = 6
    p['pyr_scale'] = pyr_scale
    eng = engine.Engine(W, H, p, max_pairs=1)
    rng = np.random.default_rng(W + H)
    frames = torch.from_numpy(rng.integers(0, 256, size=(2, H, W), dtype=np.uint8)).to(eng.device)

    def images(sweep):
        eng.set_tuning(pyr_sweep=sweep)
        flow = eng.farneback(frames, pair_stride=2)
        torch.cuda.synchronize()
        eng._keep_alive = (frames, flow)
        return [eng.tap('img', lvl, j).cpu().numpy() for lvl in range(1, len(eng.levels)) for j in (0, 1)], \
            flow.cpu().numpy()

    ref, flow_ref = images(0)
    assert len(ref) >= 4
    for sweep in (1, 2, 5, 64):
        got, flow = images(sweep)
        for k, (a, b) in enumerate(zip(ref, got)):
            assert np.array_equal(a, b), (sweep, 1 + k // 2, k % 2, float(np.abs(a - b).max()))
        assert np.array_equal(flow, flow_ref), sweep
    eng.close()
