"""Processor.run_detection with the reference's API (/root/reference/src/processor.py:21-39,277-402) on
the CUDA path.

The reference's loop handles one frame per iteration on the host.  Here the same per-frame work —
derotate (processor.py:306), FoE (:319), phi (:323), the two masks (:333-341) and the reductions behind
FrameResult (:343-362) — runs on the device for a whole batch of frames per call, through the C ABI's
mavd_detect_host (flow from Dataset.get_flow_uv, the reference's seam) or mavd_submit_host (Farneback flow
computed on the device from the frames, the new path).  Sample indices for the FoE are drawn on the host
from the global legacy NumPy generator in frame order, so the random stream is the reference's.

Out of scope (SURVEY.md §2): the homography branch (:286-303), PNG / mp4 / imshow output (:364-392, :60-81)
and the dataset-conversion methods.  The per-frame JSON (:83-84) is written when the dataset has a
results_path and write_results is true."""
from __future__ import annotations

import json
import os
from typing import Any, Dict, List, NamedTuple, Optional, Tuple

import numpy as np

from . import utils
from ._lib import HOST_SLOTS
from .detector import Detector
from .focus_of_expansion import FocusOfExpansion
from .frame_result import FrameResult
from .run_config import RunConfig


def _ratio(a: int, b: int) -> float:
    """true_positives / positives with NumPy's scalar semantics (nan for 0/0, inf for x/0)."""
    with np.errstate(divide='ignore', invalid='ignore'):
        return float(np.float64(a) / np.float64(b))


def eng_records_dtype() -> np.dtype:
    from .engine import RECORD_DTYPE
    return RECORD_DTYPE


def to_gray(frame: np.ndarray) -> np.ndarray:
    """Validates a frame: (H, W) gray or (H, W, 3) BGR uint8.  No conversion happens on the host: BGR frames are
    converted on the device (mavd_bgr2gray)."""
    if frame.ndim == 2 or (frame.ndim == 3 and frame.shape[2] == 3):
        return frame
    raise ValueError('frames must be (H, W) gray or (H, W, 3) BGR uint8')


class Detection(NamedTuple):
    """One component of a frame's estimate_fixed mask (include/mavd.h: mavd_detection): box (left, top, width,
    height), area in pixels, centroid (x, y) and the mean derotated flow (u, v) over its pixels."""
    label: int
    box: Tuple[int, int, int, int]
    area: int
    centroid: Tuple[float, float]
    flow: Tuple[float, float]


def detections_from_table(table: np.ndarray) -> List[Detection]:
    """The used entries of one frame's (max_det,) DETECTION_DTYPE table, largest component first."""
    out = []
    for d in table:
        if d['label'] == 0:
            break
        a = int(d['area'])
        out.append(Detection(int(d['label']), tuple(int(v) for v in d['box']), a,
                             (int(d['sum_x']) / a, int(d['sum_y']) / a),
                             (float(d['flow_sum'][0]) / a, float(d['flow_sum'][1]) / a)))
    return out


class Processor:
    """Acts as detector over one sequence (the dataset-conversion half of the reference class is out of scope)."""

    def __init__(self, config: RunConfig, flow_source: str = 'dataset', batch_frames: int = 8,
                 farneback_params: Optional[Dict] = None, engine: Any = None, write_results: bool = True,
                 flow_cache: Any = None, max_detections: int = 0) -> None:
        if flow_source not in ('dataset', 'farneback'):
            raise ValueError("flow_source must be 'dataset' or 'farneback'")
        self.config = config
        self.logger = self.config.logger
        self.sequence = config.sequence
        self.debug_mode = config.debug
        self.headless = config.headless
        self.dataset = config.get_dataset()
        self.flow_source = flow_source
        self.batch_frames = int(batch_frames)
        self.write_results = write_results
        # flow_source 'farneback' + flow_cache (a flow_cache.FloCache): every computed flow field is also written as
        # <cache dir>/<frame index:06d>.flo, the files Dataset.get_flow_uv reads (datasets/dataset.py:205-212)
        self.flow_cache = flow_cache
        # max_detections > 0: run_detection also lists each frame's max_detections largest components of
        # estimate_fixed in self.detections[frame index] (Detection objects, largest first)
        self.max_detections = int(max_detections)
        if not 0 <= self.max_detections <= 256:
            raise ValueError('max_detections must be in 0..256')
        self.detections: Dict[int, List[Detection]] = dict()
        width, height = self.dataset.capture_size
        if engine is None:
            from . import engine as engine_mod
            engine = engine_mod.shared_engine(width, height, farneback_params, max_pairs=self.batch_frames)
        self.engine = engine
        self.detector = Detector(self.dataset, engine=engine)
        self.detection_results: Dict[int, FrameResult] = dict()
        self.use_gt_of = False
        self.frame_step_size = 1
        self.frame_index, self.start_frame = 0, 100
        self.is_exiting = False
        self.focus_of_expansion = FocusOfExpansion(self.detector.lucas_kanade, engine=engine)
        self._pending_frame: Optional[np.ndarray] = None
        self._staging: Dict[Any, Any] = {}

    # ------------------------------------------------------------------------------------------------
    def is_active(self) -> bool:
        """Returns whether the process is still active (processor.py:56-58)."""
        return self.frame_index < self.dataset.N - 1 and not self.is_exiting

    def write(self, frame_index: int) -> None:
        """The JSON half of Processor.write (processor.py:83-84); the video/imshow half is out of scope."""
        path = getattr(self.dataset, 'results_path', None)
        if not self.write_results or not path:
            return
        utils.create_if_not_exists(path)
        with open(f'{path}/image_{frame_index:05d}.json', 'w') as f:
            f.write(json.dumps(utils.get_json(self.config.results[frame_index]), indent=4, sort_keys=True))

    # ------------------------------------------------------------------------------------------------
    def _next_frame(self) -> np.ndarray:
        """The next frame as the dataset delivers it: (H, W) gray or (H, W, 3) BGR.  BGR frames travel to the device
        unchanged and are converted there (mavd_submit_host with MAVD_HOST_BGR), as cv2.cvtColor does at
        farneback.py:74."""
        frame = self.dataset.get_frame()
        if frame is None:
            raise ValueError('Could not load frame.')
        return to_gray(np.ascontiguousarray(frame))

    def _pinned(self, slot: int, name: str, shape, dtype) -> np.ndarray:
        """A pinned host array owned by staging slot `slot`, reused from batch to batch: asynchronous copies from / to
        pageable memory are staged synchronously by the driver, which would serialise the three-stage pipeline."""
        import torch
        key = (slot, name)
        dtype = np.dtype(dtype)
        need = int(np.prod(shape)) * dtype.itemsize
        buf = self._staging.get(key)
        if buf is None or buf.numel() < need:
            buf = torch.empty((max(need, 1),), dtype=torch.uint8, pin_memory=True)
            self._staging[key] = buf
        return buf.numpy()[:need].view(dtype).reshape(shape)

    def _host_inputs(self, indices: List[int], slot: int):
        """Per-frame host inputs in frame order, in the slot's pinned staging: IMU, FoE sample indices, sky and
        segmentation masks and, when the dataset has one, the ground-truth flow (processor.py:309)."""
        from . import engine as engine_mod
        width, height = self.dataset.capture_size
        n = len(indices)
        ang, dt, rot = np.zeros((n, 3)), np.ones(n), []
        samples = self._pinned(slot, 'samples', (n, 4 * 1000), np.int32)
        sky = self._pinned(slot, 'sky', (n, height, width), np.uint8)
        seg = self._pinned(slot, 'seg', (n, height, width), np.uint8)
        gt = None
        for k, i in enumerate(indices):
            a, d, on = self.detector.imu_for(i - self.frame_step_size, i)
            ang[k], dt[k] = a, d
            rot.append(on)
            samples[k] = FocusOfExpansion.draw_sample_indices(height, width)     # global RNG, frame order
            sky[k] = np.asarray(self.dataset.get_sky_segmentation(i)).astype(np.uint8)
            s = np.asarray(self.dataset.get_segmentation(i))
            seg[k] = s[..., 0] if s.ndim == 3 else s
            g = self.dataset.get_gt_of(i) if hasattr(self.dataset, 'get_gt_of') else None
            if g is not None:
                if gt is None:
                    gt = self._pinned(slot, 'gt_flow', (n, height, width, 2), np.float32)
                    gt[:k] = 0.0
                gt[k] = g
            elif gt is not None:
                gt[k] = 0.0
        return engine_mod.make_imu(n, ang, dt, derotate=rot), samples, sky, seg, gt

    def _frame_result(self, i: int, rec: np.void, sky_k: np.ndarray, has_gt: bool = False) -> FrameResult:
        """processor.py:327-329,343-362 from the device record of frame i."""
        st = rec['stats']
        fr = FrameResult()
        foe = (rec['foe'][0], rec['foe'][1])
        fr.foe_dense = (0.0, 0.0) if (foe[0] == 0.0 and foe[1] == 0.0) else foe
        foe_gt = self.dataset.get_gt_foe(i)
        assert foe_gt is not None
        fr.foe_gt = foe_gt
        x0, y0, x1, y1 = (int(v) for v in st['seg_bbox'])
        center = utils.Rectangle.from_points((x0, y0), (x1, y1)).get_center()
        fr.center_phi = np.rad2deg(np.arctan2(center[1] - fr.foe_gt[1], center[0] - fr.foe_gt[0]))
        fr.tpr = _ratio(st['tp_total'], st['positives'])
        fr.fpr = _ratio(st['fp_total'], st['negatives'])
        fr.tpr_fixed = _ratio(st['tp_fixed'], st['positives'])
        fr.fpr_fixed = _ratio(st['fp_fixed'], st['negatives'])
        depth = self.dataset.get_depth(i) if hasattr(self.dataset, 'get_depth') else None
        if depth is not None and hasattr(self.dataset, 'validate_sky_segment'):
            fr.sky_tpr, fr.sky_fpr = self.dataset.validate_sky_segment(sky_k.astype(bool), depth)
        fr.drone_size_pixels = int(st['positives'])
        fr.time = self.dataset.get_time(i)
        fr.drone_flow_pixels = self._drone_flow_gt(i, rec, has_gt)
        return fr

    def _drone_flow_gt(self, i: int, rec: np.void, has_gt: bool) -> Tuple[float, float]:
        """np.average(gt_flow_uv_derotated[segmentation > 127]) (processor.py:344,359).  The ground-truth flow of the
        whole batch went to the device with the batch (mavd_aux_inputs.gt_flow) and was derotated and summed there;
        without a ground-truth flow the estimated flow's average over the segmentation is reported."""
        st = rec['stats']
        pos = int(st['positives'])
        s = st['gt_flow_sum'] if has_gt else st['seg_flow_sum']
        return (_ratio(s[0], pos), _ratio(s[1], pos)) if pos else (float('nan'), float('nan'))

    # ------------------------------------------------------------------------------------------------
    def run_detection(self) -> Dict[int, FrameResult]:
        """Runs the detection (processor.py:277-396), a batch of frames per device call."""
        if self.detector.is_homography_based():
            raise NotImplementedError('the homography branch is outside the rebuilt hot path (SURVEY.md §2)')
        eng = self.engine
        width, height = self.dataset.capture_size
        B = self.batch_frames
        inflight: List[tuple] = []   # (slot, indices, records, sky, gt?, flow, detection tables)
        slot = 0
        D = self.max_detections

        def det_tables(s: int, n: int) -> Optional[np.ndarray]:
            from .engine import DETECTION_DTYPE
            return self._pinned(s, 'detections', (n, D), DETECTION_DTYPE) if D else None

        def finish(entry) -> None:
            s, indices, records, sky, has_gt, flow, det = entry
            if s >= 0:
                eng.wait_host(s)
            if flow is not None:
                for k, i in enumerate(indices):           # frame_step_size may skip indices: one file per frame
                    self.flow_cache.put_batch(i, flow[k:k + 1])
            if det is not None:
                for k, i in enumerate(indices):
                    self.detections[i] = detections_from_table(det[k])
            for k, i in enumerate(indices):
                fr = self._frame_result(i, records[k], sky[k], has_gt)
                self.detection_results[i] = fr
                self.config.results[i] = fr
                self.write(i)

        while self.is_active():
            first = self.frame_index
            indices = list(range(first, min(first + B * self.frame_step_size, self.dataset.N - 1), self.frame_step_size))
            n = len(indices)
            if self.flow_source == 'dataset':
                for _ in indices:
                    self.dataset.get_frame()                      # keeps the capture in step (processor.py:284)
                flows = self._pinned(0, 'flow', (n, height, width, 2), np.float32)
                for k, i in enumerate(indices):
                    f = self.dataset.get_flow_uv(i)
                    if f is None:
                        raise ValueError('Could not load flow field.')
                    flows[k] = f
                imu, samples, sky, seg, gt = self._host_inputs(indices, 0)
                records = self._pinned(0, 'records', (n,), eng_records_dtype())
                det = det_tables(0, n)
                self.focus_of_expansion._eng()                   # its FoE thresholds -> eng.detect_params (shared engine)
                eng.detect_host(flows, imu, samples, sky=sky, seg=seg, gt_flow=gt, records=records, detections=det)
                finish((-1, indices, records, sky, gt is not None, None, det))
            else:
                # flow(i) = Farneback(frame i, frame i+1); consecutive batches share one frame
                if len(inflight) == HOST_SLOTS - 1:
                    finish(inflight.pop(0))                      # frees the staging of the slot used next
                first_frame = self._pending_frame if self._pending_frame is not None else self._next_frame()
                frames = self._pinned(slot, 'frames', (n + 1,) + first_frame.shape, np.uint8)     # gray or BGR, as delivered
                frames[0] = first_frame
                for k in range(n):
                    frames[k + 1] = self._next_frame()
                self._pending_frame = frames[-1].copy()
                imu, samples, sky, seg, gt = self._host_inputs(indices, slot)
                records = self._pinned(slot, 'records', (n,), eng_records_dtype())
                flow = self._pinned(slot, 'flow_out', (n, height, width, 2), np.float32) if self.flow_cache is not None \
                    else None
                det = det_tables(slot, n)
                self.focus_of_expansion._eng()                   # the call copies detect_params: batches in flight keep theirs
                eng.submit_host(slot, frames, imu, samples, n_pairs=n, sky=sky, seg=seg, gt_flow=gt, flow_out=flow,
                                records=records, detections=det)
                inflight.append((slot, indices, records, sky, gt is not None, flow, det))
                slot = (slot + 1) % HOST_SLOTS
            self.frame_index = indices[-1] + self.frame_step_size
            n10 = int(self.dataset.N / 10)
            if n10 and self.logger is not None and (self.frame_index // n10) != (first // n10):
                self.logger.info(f'{self.frame_index / self.dataset.N * 100:.2f}% {self.frame_index} / {self.dataset.N}')
        while inflight:
            finish(inflight.pop(0))
        return self.detection_results

    def release(self) -> None:
        """Release all media resources (processor.py:398-402)."""
        if hasattr(self.dataset, 'release'):
            self.dataset.release()
