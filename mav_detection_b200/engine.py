"""Thin host wrapper over the C ABI: owns one mavd handle and passes torch CUDA tensors' data pointers
and the current CUDA stream to libmavd.  PyTorch is plumbing here (device memory, streams,
torch.distributed) — all compute runs in the hand-written sm_100a kernels of csrc/."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import AuxInputs, Config, DetectParams, Detection, FarnebackParams, FrameRecord, FrameStats, Imu, Tuning, check

# cv2.calcOpticalFlowFarneback arguments used by the reference (src/farneback.py:78-80)
REFERENCE_PARAMS = dict(pyr_scale=0.4, levels=1, winsize=12, iterations=10, poly_n=8, poly_sigma=1.2, flags=0)
# OpenCV's documented sample values (BASELINE config 2)
SAMPLE_PARAMS = dict(pyr_scale=0.5, levels=5, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2, flags=0)

RECORD_DTYPE = np.dtype(FrameRecord)
STATS_DTYPE = np.dtype(FrameStats)
DETECTION_DTYPE = np.dtype(Detection)


def make_imu(n: int, ang: Optional[np.ndarray] = None, dt=None, derotate=None) -> C.Array:
    """Build the mavd_imu array for n frames.  ang (n,3), dt (n,) or scalar, derotate (n,) bool."""
    arr = (Imu * n)()
    for i in range(n):
        a = (0.0, 0.0, 0.0) if ang is None else np.asarray(ang, np.float64).reshape(-1, 3)[i]
        arr[i].ang[0], arr[i].ang[1], arr[i].ang[2] = float(a[0]), float(a[1]), float(a[2])
        arr[i].dt = float(dt if np.isscalar(dt) else (1.0 if dt is None else dt[i]))
        d = True if derotate is None else (derotate if isinstance(derotate, (bool, int)) else derotate[i])
        arr[i].derotate = 1 if d else 0
    return arr


def parse_tuning(text: str) -> Dict[str, int]:
    """'pyr_sweep=8,use_graph=0' -> {'pyr_sweep': 8, 'use_graph': 0} (bench.py --tune, tools/gpu_ab.sh)."""
    out: Dict[str, int] = {}
    names = {f[0] for f in Tuning._fields_} - {'reserved'}
    for item in filter(None, (t.strip() for t in text.split(','))):
        k, _, v = item.partition('=')
        if k not in names:
            raise ValueError('unknown tuning field %r (known: %s)' % (k, ', '.join(sorted(names))))
        out[k] = int(v)
    return out


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _hp(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


class Engine:
    """One handle per (device, W, H, Farneback parameters) — SURVEY.md §8b threading/state."""

    def __init__(self, width: int, height: int, params: Optional[Dict] = None, max_pairs: int = 1,
                 device: int = 0) -> None:
        if not torch.cuda.is_available():
            raise _lib.MavdError('no CUDA device: the mav-detection hot path has no CPU fallback')
        self.lib = _lib.load()
        p = dict(REFERENCE_PARAMS)
        if params:
            p.update(params)
        self.params = p
        self.width, self.height, self.max_pairs = int(width), int(height), int(max_pairs)
        self.device = torch.device('cuda', device)
        cfg = Config(device, self.width, self.height, self.max_pairs,
                     FarnebackParams(float(p['pyr_scale']), int(p['levels']), int(p['winsize']),
                                     int(p['iterations']), int(p['poly_n']), float(p['poly_sigma']),
                                     int(p['flags'])))
        h = C.c_void_p()
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)  # make sure the primary context exists
            check(self.lib.mavd_create(C.byref(cfg), C.byref(h)))
        self._h = h
        n = C.c_int32()
        ws, hs = (C.c_int32 * 16)(), (C.c_int32 * 16)()
        check(self.lib.mavd_level_info(self._h, C.byref(n), ws, hs))
        self.levels: List[Tuple[int, int]] = [(ws[i], hs[i]) for i in range(n.value)]
        self.detect_params = DetectParams()
        self.lib.mavd_default_detect_params(C.byref(self.detect_params))
        self._inflight: Dict[int, tuple] = {}
        self._open_streams: set = set()
        # counts the non-stream Farneback calls made through this engine: each one ends every frame stream
        self.stream_epoch = 0

    # -- lifecycle --------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, '_h', None) is not None and self._h.value:
            self.lib.mavd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def workspace_bytes(self) -> int:
        out = C.c_size_t()
        check(self.lib.mavd_workspace_bytes(self._h, C.byref(out)))
        return out.value

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- launch-shape tuning (never changes results) --------------------------------------------
    def get_tuning(self) -> Dict[str, int]:
        t = Tuning()
        check(self.lib.mavd_get_tuning(self._h, C.byref(t)))
        return {f[0]: int(getattr(t, f[0])) for f in Tuning._fields_ if f[0] != 'reserved'}

    def set_tuning(self, **fields: int) -> None:
        """Set mavd_tuning fields by name; the handle must be idle (the call synchronises the device)."""
        t = Tuning()
        check(self.lib.mavd_get_tuning(self._h, C.byref(t)))
        for k, v in fields.items():
            if k == 'reserved' or not hasattr(t, k):
                raise ValueError('unknown tuning field %r' % k)
            setattr(t, k, int(v))
        check(self.lib.mavd_set_tuning(self._h, C.byref(t)))

    def _check_samples(self, samples: torch.Tensor, n: int) -> None:
        if not isinstance(samples, torch.Tensor) or samples.dtype != torch.int32 or not samples.is_cuda or \
                samples.device != self.device or not samples.is_contiguous() or \
                tuple(samples.shape) != (n, _lib.SAMPLES_PER_FRAME):
            raise ValueError('samples must be a contiguous int32 tensor (%d, %d) on %s: [ry(2000) | rx(2000)] per frame'
                             % (n, _lib.SAMPLES_PER_FRAME, self.device))

    def _aux(self, sky, seg, gt_flow, n: int, host: bool = False, sky_packed: bool = False,
             seg_packed: bool = False) -> AuxInputs:
        """mavd_aux_inputs from optional sky / seg masks ((H, W) shared or (n, H, W) per frame; packed: (bytes,) or
        (n, bytes)) and an optional (n, H, W, 2) float32 ground-truth flow; device tensors or host arrays."""
        npx = self.width * self.height
        pb = self.packed_mask_bytes

        def one(t, packed, name):
            if t is None:
                return None, 0
            if host:
                if t.dtype not in (np.uint8, np.bool_) or not t.flags['C_CONTIGUOUS']:
                    raise ValueError('%s must be a C-contiguous uint8/bool array' % name)
                dim, size, ptr = t.ndim, t.size, t.ctypes.data
            else:
                if t.dtype not in (torch.uint8, torch.bool) or not t.is_cuda or not t.is_contiguous():
                    raise ValueError('%s must be a contiguous CUDA uint8/bool tensor' % name)
                dim, size, ptr = t.dim(), t.numel(), t.data_ptr()
            per, shared_dim = (pb, 1) if packed else (npx, 2)
            if dim == shared_dim and size == per:
                return ptr, 0
            if dim == shared_dim + 1 and size == per * n:
                return ptr, per
            raise ValueError('%s has %d elements: expected %d (shared) or %d x %d (per frame)' % (name, size, per, n, per))
        a = AuxInputs()
        a.sky, a.sky_stride = one(sky, sky_packed, 'sky')
        a.seg, a.seg_stride = one(seg, seg_packed, 'seg')
        if gt_flow is not None:
            if host:
                ok = gt_flow.dtype == np.float32 and gt_flow.flags['C_CONTIGUOUS'] and \
                    tuple(gt_flow.shape) == (n, self.height, self.width, 2)
                a.gt_flow = gt_flow.ctypes.data if ok else None
            else:
                ok = gt_flow.dtype == torch.float32 and gt_flow.is_cuda and gt_flow.is_contiguous() and \
                    tuple(gt_flow.shape) == (n, self.height, self.width, 2)
                a.gt_flow = gt_flow.data_ptr() if ok else None
            if not ok:
                raise ValueError('gt_flow must be contiguous float32 (%d, %d, %d, 2)' % (n, self.height, self.width))
        return a

    @property
    def packed_mask_bytes(self) -> int:
        """Bytes one (H, W) mask occupies at 1 bit per pixel on the host<->device wire."""
        return int(self.lib.mavd_packed_mask_bytes(self.width, self.height))

    def pack_mask_host(self, mask: np.ndarray) -> np.ndarray:
        """(..., H, W) uint8/bool host mask -> (..., packed_mask_bytes) uint8, the layout MAVD_HOST_*_PACKED expects
        (numpy.packbits(bitorder='little') of the flattened frame, zero padded)."""
        lead = mask.shape[:-2]
        bits = np.packbits(np.ascontiguousarray(mask).reshape(lead + (-1,)) != 0, axis=-1, bitorder='little')
        out = np.zeros(lead + (self.packed_mask_bytes,), np.uint8)
        out[..., :bits.shape[-1]] = bits
        return out

    def unpack_mask_host(self, bits: np.ndarray) -> np.ndarray:
        """The inverse: (..., packed_mask_bytes) uint8 -> (..., H, W) uint8 0/1."""
        lead = bits.shape[:-1]
        flat = np.unpackbits(bits, axis=-1, bitorder='little')[..., :self.width * self.height]
        return flat.reshape(lead + (self.height, self.width))

    def pack_mask(self, mask: torch.Tensor) -> torch.Tensor:
        """(n, H, W) CUDA uint8 mask -> (n, packed_mask_bytes) uint8 (mavd_pack_mask)."""
        mask = mask.contiguous()
        n = mask.shape[0]
        out = torch.empty((n, self.packed_mask_bytes), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.mavd_pack_mask(mask.data_ptr(), n, self.width * self.height, out.data_ptr(), self._stream()))
        return out

    def unpack_mask(self, bits: torch.Tensor, value: int = 1) -> torch.Tensor:
        """(n, packed_mask_bytes) CUDA uint8 -> (n, H, W) uint8 with set bits = value (mavd_unpack_mask)."""
        bits = bits.contiguous()
        n = bits.shape[0]
        out = torch.empty((n, self.height, self.width), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.mavd_unpack_mask(bits.data_ptr(), n, self.width * self.height, int(value), out.data_ptr(),
                                            self._stream()))
        return out

    def _check_frames(self, frames: torch.Tensor, n_pairs: int, pair_stride: int) -> None:
        need = n_pairs + 1 if pair_stride == 1 else 2 * n_pairs
        if frames.dtype != torch.uint8 or not frames.is_cuda or not frames.is_contiguous():
            raise ValueError('frames must be a contiguous CUDA uint8 tensor (F, H, W)')
        if frames.dim() != 3 or frames.shape[1] != self.height or frames.shape[2] != self.width:
            raise ValueError('frames must have shape (F, %d, %d), got %s' % (self.height, self.width,
                                                                             tuple(frames.shape)))
        if frames.shape[0] < need:
            raise ValueError('%d pairs with pair_stride %d need %d frames, got %d'
                             % (n_pairs, pair_stride, need, frames.shape[0]))

    # -- stage 0 -----------------------------------------------------------------------------
    def bgr2gray(self, bgr: torch.Tensor) -> torch.Tensor:
        """cv2.cvtColor(img, COLOR_BGR2GRAY) — src/farneback.py:74.  (..., 3) uint8 -> (...) uint8."""
        if bgr.dtype != torch.uint8 or not bgr.is_cuda or bgr.shape[-1] != 3:
            raise ValueError('bgr must be a CUDA uint8 tensor (..., 3)')
        bgr = bgr.contiguous()
        if bgr.device != self.device:
            raise ValueError('bgr lives on %s, the engine on %s' % (bgr.device, self.device))
        out = torch.empty(bgr.shape[:-1], dtype=torch.uint8, device=bgr.device)
        with torch.cuda.device(self.device):        # handle-less entry point: runs on the current device
            check(self.lib.mavd_bgr2gray(bgr.data_ptr(), out.data_ptr(), out.numel(), self._stream()))
        return out

    # -- stage 1 -----------------------------------------------------------------------------
    def farneback(self, frames: torch.Tensor, n_pairs: Optional[int] = None, pair_stride: int = 1,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Dense flow for every pair — cv2.calcOpticalFlowFarneback (src/farneback.py:76-80)."""
        if n_pairs is None:
            n_pairs = frames.shape[0] - 1 if pair_stride == 1 else frames.shape[0] // 2
        self._check_frames(frames, n_pairs, pair_stride)
        if out is None:
            out = torch.empty((n_pairs, self.height, self.width, 2), dtype=torch.float32, device=self.device)
        self.stream_epoch += 1
        check(self.lib.mavd_farneback(self._h, frames.data_ptr(), n_pairs, pair_stride, out.data_ptr(),
                                      self._stream()))
        return out

    def tap(self, kind: str, level: int, index: int = 0) -> torch.Tensor:
        kinds = {'img': (0, 1), 'R': (1, 5), 'M': (2, 5), 'flow': (3, 2)}
        k, ch = kinds[kind]
        w, h = self.levels[level]
        shape = (h, w) if ch == 1 else (h, w, ch)
        out = torch.empty(shape, dtype=torch.float32, device=self.device)
        check(self.lib.mavd_farneback_tap(self._h, k, level, index, out.data_ptr(), self._stream()))
        return out

    # -- stage 1.5 ----------------------------------------------------------------------------
    def derotate(self, flow: torch.Tensor, imu) -> torch.Tensor:
        """Detector.derotate for a batch — detector.py:70-117.  float32 or float64 (n, H, W, 2) in, float64 out."""
        n = flow.shape[0]
        kind = self._flow_kind(flow)
        out = torch.empty(flow.shape, dtype=torch.float64, device=self.device)
        fn = self.lib.mavd_derotate_f64 if kind else self.lib.mavd_derotate
        check(fn(self._h, flow.data_ptr(), n, imu, out.data_ptr(), self._stream()))
        return out

    # -- stage 2 -----------------------------------------------------------------------------
    def foe(self, flow: torch.Tensor, imu, samples: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        n = flow.shape[0]
        if samples.dtype != torch.int32 or tuple(samples.shape) != (n, _lib.SAMPLES_PER_FRAME):
            raise ValueError('samples must be int32 (n, %d): [ry(2000) | rx(2000)]' % _lib.SAMPLES_PER_FRAME)
        foe = torch.empty((n, 2), dtype=torch.float64, device=self.device)
        cnt = torch.empty((n,), dtype=torch.int32, device=self.device)
        check(self.lib.mavd_foe(self._h, flow.data_ptr(), n, imu, C.byref(self.detect_params),
                                samples.data_ptr(), foe.data_ptr(), cnt.data_ptr(), self._stream()))
        return foe, cnt

    # -- stage 3 -----------------------------------------------------------------------------
    def residual_masks(self, flow: torch.Tensor, imu, foe: torch.Tensor, sky: Optional[torch.Tensor] = None,
                       seg: Optional[torch.Tensor] = None, want_phi: bool = True, want_stats: bool = True):
        n = flow.shape[0]
        npx = self.width * self.height
        phi = torch.zeros((n, self.height, self.width), dtype=torch.float64, device=self.device) if want_phi else None
        total = torch.empty((n, self.height, self.width), dtype=torch.uint8, device=self.device)
        fixed = torch.empty_like(total)
        stats = torch.zeros((n, STATS_DTYPE.itemsize), dtype=torch.uint8, device=self.device) if want_stats else None

        def stride(t):
            if t is None:
                return 0
            if t.dtype not in (torch.uint8, torch.bool) or not t.is_contiguous():
                raise ValueError('sky/seg must be contiguous uint8/bool tensors')
            return 0 if t.dim() == 2 else npx
        check(self.lib.mavd_residual_masks(self._h, flow.data_ptr(), n, imu, C.byref(self.detect_params),
                                           foe.data_ptr(), _ptr(sky), stride(sky), _ptr(seg), stride(seg),
                                           _ptr(phi), total.data_ptr(), fixed.data_ptr(), _ptr(stats),
                                           self._stream()))
        return phi, total, fixed, stats

    # -- reference-literal seams (FocusOfExpansion methods on a flow array of either dtype) -----
    def _flow_kind(self, flow: torch.Tensor) -> int:
        if flow.dtype not in (torch.float32, torch.float64) or not flow.is_cuda or not flow.is_contiguous():
            raise ValueError('flow must be a contiguous CUDA float32/float64 tensor (n, H, W, 2)')
        if tuple(flow.shape[1:]) != (self.height, self.width, 2):
            raise ValueError('flow must have shape (n, %d, %d, 2), got %s' % (self.height, self.width, tuple(flow.shape)))
        return 1 if flow.dtype == torch.float64 else 0

    def foe_dense(self, flow: torch.Tensor, samples: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """FocusOfExpansion.get_FOE_dense(flow_uv) on the flow as given (no IMU) — focus_of_expansion.py:56-86."""
        n = flow.shape[0]
        if samples.dtype != torch.int32 or tuple(samples.shape) != (n, _lib.SAMPLES_PER_FRAME):
            raise ValueError('samples must be int32 (n, %d): [ry(2000) | rx(2000)]' % _lib.SAMPLES_PER_FRAME)
        foe = torch.empty((n, 2), dtype=torch.float64, device=self.device)
        cnt = torch.empty((n,), dtype=torch.int32, device=self.device)
        check(self.lib.mavd_foe_dense(self._h, flow.data_ptr(), self._flow_kind(flow), n, C.byref(self.detect_params),
                                      samples.data_ptr(), foe.data_ptr(), cnt.data_ptr(), self._stream()))
        return foe, cnt

    def ransac(self, estimates: torch.Tensor, threshold: Optional[float] = None) -> torch.Tensor:
        """FocusOfExpansion.ransac(estimates) — focus_of_expansion.py:32-54.  (K, 2) float64 -> (2,) float64."""
        if estimates.dtype != torch.float64 or estimates.dim() != 2 or estimates.shape[1] != 2:
            raise ValueError('estimates must be a (K, 2) float64 tensor')
        estimates = estimates.contiguous()
        out = torch.empty((2,), dtype=torch.float64, device=self.device)
        thr = self.detect_params.ransac_threshold if threshold is None else float(threshold)
        check(self.lib.mavd_ransac(self._h, estimates.data_ptr() if estimates.shape[0] else None, estimates.shape[0],
                                   thr, out.data_ptr(), self._stream()))
        return out

    def get_phi(self, flow: torch.Tensor, foe: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """FocusOfExpansion.get_phi(flow, FoE) — focus_of_expansion.py:150-184.  Returns (phi in the flow's
        dtype, per-frame max phi = the max_flow side effect)."""
        n = flow.shape[0]
        kind = self._flow_kind(flow)
        phi = torch.empty((n, self.height, self.width), dtype=flow.dtype, device=self.device)
        mx = torch.empty((n,), dtype=torch.float64, device=self.device)
        foe = foe.to(device=self.device, dtype=torch.float64).contiguous()
        if kind == 0:
            # the C ABI lays float32 phi at the front of each frame's 8-byte-per-pixel slot
            buf = torch.empty((n, self.height, self.width), dtype=torch.float64, device=self.device)
            check(self.lib.mavd_get_phi(self._h, flow.data_ptr(), 0, n, foe.data_ptr(), buf.data_ptr(), mx.data_ptr(),
                                        self._stream()))
            npx = self.height * self.width
            phi = buf.view(torch.float32).view(n, 2 * npx)[:, :npx].reshape(n, self.height, self.width).clone()
        else:
            check(self.lib.mavd_get_phi(self._h, flow.data_ptr(), 1, n, foe.data_ptr(), phi.data_ptr(), mx.data_ptr(),
                                        self._stream()))
        return phi, mx

    # -- stage 4 -----------------------------------------------------------------------------
    def ccl(self, mask: torch.Tensor, max_boxes: int = _lib.MAX_BOXES, want_labels: bool = True):
        n = mask.shape[0]
        labels = torch.empty((n, self.height, self.width), dtype=torch.int32, device=self.device) if want_labels else None
        boxes = torch.zeros((n, max_boxes, 5), dtype=torch.int32, device=self.device)
        cnt = torch.empty((n,), dtype=torch.int32, device=self.device)
        check(self.lib.mavd_ccl(self._h, mask.data_ptr(), n, _ptr(labels), boxes.data_ptr(), max_boxes,
                                cnt.data_ptr(), self._stream()))
        return labels, boxes, cnt

    def _det_count(self, max_det) -> int:
        if isinstance(max_det, bool) or not isinstance(max_det, (int, np.integer)) or \
                not 1 <= int(max_det) <= _lib.MAX_DETECTIONS:
            raise ValueError('max_det must be an int in 1..%d' % _lib.MAX_DETECTIONS)
        return int(max_det)

    def _det_device(self, detections: Optional[int], n: int) -> Tuple[int, Optional[torch.Tensor]]:
        """(max_det, table) for a device call asked for `detections` entries per frame: an (n, max_det, itemsize) uint8
        CUDA tensor, or (0, None) for no table."""
        if detections is None:
            return 0, None
        max_det = self._det_count(detections)
        return max_det, torch.empty((n, max_det, DETECTION_DTYPE.itemsize), dtype=torch.uint8, device=self.device)

    def _det_host(self, det: Optional[np.ndarray], n: int) -> Tuple[int, Optional[int]]:
        """(max_det, pointer) of a host detection table: (n, max_det) DETECTION_DTYPE, C-contiguous (pinned for the
        copy to be asynchronous)."""
        if det is None:
            return 0, None
        if not isinstance(det, np.ndarray) or det.dtype != DETECTION_DTYPE or det.ndim != 2 or det.shape[0] < n or \
                not det.flags['C_CONTIGUOUS']:
            raise ValueError('detections must be a C-contiguous (n, max_det) array of DETECTION_DTYPE')
        return self._det_count(det.shape[1]), det.ctypes.data

    def detections(self, mask: torch.Tensor, flow: Optional[torch.Tensor] = None, imu=None,
                   max_det: int = 32) -> torch.Tensor:
        """Detection table of every (H, W) mask of an (n, H, W) uint8/bool CUDA tensor (non-zero = foreground): the
        max_det largest 8-connected components by (area desc, label asc).  With a float32 (n, H, W, 2) flow and its imu
        array, flow_sum is the derotated flow summed over each component.  Returns an (n, max_det, itemsize) uint8
        CUDA tensor of mavd_detection (detections_to_numpy)."""
        max_det = self._det_count(max_det)
        if mask.dtype not in (torch.uint8, torch.bool) or not mask.is_cuda or not mask.is_contiguous() or \
                tuple(mask.shape[1:]) != (self.height, self.width):
            raise ValueError('mask must be a contiguous CUDA uint8/bool tensor (n, %d, %d)' % (self.height, self.width))
        n = mask.shape[0]
        if flow is not None:
            if self._flow_kind(flow) != 0 or flow.shape[0] != n:
                raise ValueError('flow must be float32 (%d, %d, %d, 2)' % (n, self.height, self.width))
            if imu is None:
                raise ValueError('a flow needs its imu array')
        out = torch.empty((n, max_det, DETECTION_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        check(self.lib.mavd_detections(self._h, mask.data_ptr(), n, _ptr(flow), imu, max_det, out.data_ptr(),
                                       self._stream()))
        return out

    @staticmethod
    def detections_to_numpy(det: torch.Tensor) -> np.ndarray:
        """(n, max_det, itemsize) uint8 tensor -> (n, max_det) DETECTION_DTYPE array."""
        return det.cpu().numpy().view(DETECTION_DTYPE)[..., 0]

    # -- sparse features -------------------------------------------------------------------------
    def _check_u8_frames(self, frames: torch.Tensor, n: int, what: str) -> None:
        if frames.dtype != torch.uint8 or not frames.is_cuda or not frames.is_contiguous() or frames.dim() != 3 or \
                tuple(frames.shape[1:]) != (self.height, self.width) or frames.shape[0] < n:
            raise ValueError('%s must be a contiguous CUDA uint8 tensor (>= %d, %d, %d)' % (what, n, self.height,
                                                                                            self.width))

    def good_features(self, frames: torch.Tensor, max_corners: int, quality_level: float, min_distance: float,
                      block_size: int = 3, mask: Optional[torch.Tensor] = None, want_eig: bool = False):
        """cv2.goodFeaturesToTrack(frame, max_corners, quality_level, min_distance, mask, block_size) for every frame
        of an (n, H, W) uint8 CUDA tensor.  Returns (corners (n, max_corners, 2) float32, counts (n,) int32[, eig
        (n, H, W) float32]).  counts are not limited by max_corners; frame i's corners are corners[i, :min(count,
        max_corners)] in cv2's order.  mask: (H, W) for every frame or (n, H, W), uint8 or bool."""
        n = frames.shape[0]
        self._check_u8_frames(frames, n, 'frames')
        prm = _lib.GfttParams(int(max_corners), float(quality_level), float(min_distance), int(block_size), 3)
        stride = 0
        if mask is not None:
            if mask.dtype not in (torch.uint8, torch.bool) or not mask.is_cuda or not mask.is_contiguous() or \
                    tuple(mask.shape[-2:]) != (self.height, self.width) or mask.dim() not in (2, 3) or \
                    (mask.dim() == 3 and mask.shape[0] != n):
                raise ValueError('mask must be a contiguous CUDA uint8/bool tensor (H, W) or (n, H, W)')
            stride = self.width * self.height if mask.dim() == 3 else 0
        corners = torch.zeros((n, max(int(max_corners), 0), 2), dtype=torch.float32, device=self.device)
        counts = torch.zeros((n,), dtype=torch.int32, device=self.device)
        eig = torch.empty((n, self.height, self.width), dtype=torch.float32, device=self.device) if want_eig else None
        check(self.lib.mavd_good_features_to_track(self._h, frames.data_ptr(), n, C.byref(prm), _ptr(mask), stride,
                                                   corners.data_ptr() if corners.numel() else None, counts.data_ptr(),
                                                   _ptr(eig), self._stream()))
        return (corners, counts, eig) if want_eig else (corners, counts)

    def pyr_lk(self, frames: torch.Tensor, prev_pts: torch.Tensor, n_points: Optional[torch.Tensor] = None,
               pair_stride: int = 1, win: Tuple[int, int] = (21, 21), max_level: int = 3,
               criteria: Tuple[int, int, float] = (_lib.TERM_COUNT | _lib.TERM_EPS, 30, 0.01), flags: int = 0,
               min_eig_threshold: float = 1e-4):
        """cv2.calcOpticalFlowPyrLK(prev, next, prevPts, None, win, max_level, criteria, flags, min_eig_threshold) for
        every pair: pair p tracks prev_pts[p] ((n_pairs, N, 2) float32 CUDA) from frame p*pair_stride to the next
        frame.  n_points: optional (n_pairs,) int32 counts (good_features' counts).  Returns (next_pts (n_pairs, N, 2)
        float32, status (n_pairs, N) uint8, err (n_pairs, N) float32)."""
        if prev_pts.dtype != torch.float32 or not prev_pts.is_cuda or not prev_pts.is_contiguous() or \
                prev_pts.dim() != 3 or prev_pts.shape[2] != 2:
            raise ValueError('prev_pts must be a contiguous CUDA float32 tensor (n_pairs, N, 2)')
        n_pairs, n = prev_pts.shape[0], prev_pts.shape[1]
        if pair_stride not in (1, 2):
            raise ValueError('pair_stride must be 1 or 2')
        self._check_u8_frames(frames, (n_pairs - 1) * pair_stride + 2 if n_pairs else 0, 'frames')
        if n_points is not None and (n_points.dtype != torch.int32 or not n_points.is_cuda or
                                     not n_points.is_contiguous() or n_points.shape[0] < n_pairs):
            raise ValueError('n_points must be a contiguous CUDA int32 tensor (>= n_pairs,)')
        prm = _lib.LkParams(int(win[0]), int(win[1]), int(max_level), int(criteria[0]), int(criteria[1]),
                            float(criteria[2]), int(flags), float(min_eig_threshold))
        nxt = torch.empty_like(prev_pts)
        status = torch.empty((n_pairs, n), dtype=torch.uint8, device=self.device)
        err = torch.empty((n_pairs, n), dtype=torch.float32, device=self.device)
        check(self.lib.mavd_pyr_lk(self._h, frames.data_ptr(), n_pairs, pair_stride, C.byref(prm), prev_pts.data_ptr(),
                                   n, _ptr(n_points), nxt.data_ptr(), status.data_ptr(), err.data_ptr(),
                                   self._stream()))
        return nxt, status, err

    # -- whole path ----------------------------------------------------------------------------
    def process(self, frames: torch.Tensor, imu, samples: torch.Tensor, n_pairs: Optional[int] = None,
                pair_stride: int = 1, sky: Optional[torch.Tensor] = None, seg: Optional[torch.Tensor] = None,
                flow_out: Optional[torch.Tensor] = None, total_out: Optional[torch.Tensor] = None,
                fixed_out: Optional[torch.Tensor] = None, records: Optional[torch.Tensor] = None,
                gt_flow: Optional[torch.Tensor] = None, detections: Optional[int] = None):
        """Farneback -> derotate -> FoE -> phi/masks -> components, device buffers in and out.
        Returns the (n_pairs, sizeof(mavd_frame_record)) uint8 CUDA tensor of records; with detections = max_det,
        (records, the (n_pairs, max_det, itemsize) uint8 CUDA tensor of each pair's detection table)."""
        if n_pairs is None:
            n_pairs = frames.shape[0] - 1 if pair_stride == 1 else frames.shape[0] // 2
        self._check_frames(frames, n_pairs, pair_stride)
        self._check_samples(samples, n_pairs)
        if records is None:
            records = torch.empty((n_pairs, RECORD_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        aux = self._aux(sky, seg, gt_flow, n_pairs)
        max_det, det = self._det_device(detections, n_pairs)
        self.stream_epoch += 1
        check(self.lib.mavd_process(self._h, frames.data_ptr(), n_pairs, pair_stride, imu, C.byref(self.detect_params),
                                    samples.data_ptr(), C.byref(aux), _ptr(flow_out), _ptr(total_out), _ptr(fixed_out),
                                    records.data_ptr(), max_det, _ptr(det), self._stream()))
        return records if det is None else (records, det)

    def detect(self, flow: torch.Tensor, imu, samples: torch.Tensor, sky: Optional[torch.Tensor] = None,
               seg: Optional[torch.Tensor] = None, total_out: Optional[torch.Tensor] = None,
               fixed_out: Optional[torch.Tensor] = None, records: Optional[torch.Tensor] = None,
               gt_flow: Optional[torch.Tensor] = None, detections: Optional[int] = None):
        """derotate -> FoE -> phi/masks -> components from a given float32 flow (the Dataset.get_flow_uv seam).
        detections = max_det: returns (records, detection tables) as process does."""
        n = flow.shape[0]
        if flow.dtype != torch.float32 or not flow.is_cuda or not flow.is_contiguous() or \
                tuple(flow.shape[1:]) != (self.height, self.width, 2):
            raise ValueError('flow must be a contiguous CUDA float32 tensor (n, %d, %d, 2)' % (self.height, self.width))
        self._check_samples(samples, n)
        if records is None:
            records = torch.empty((n, RECORD_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        aux = self._aux(sky, seg, gt_flow, n)
        max_det, det = self._det_device(detections, n)
        check(self.lib.mavd_detect(self._h, flow.data_ptr(), n, imu, C.byref(self.detect_params), samples.data_ptr(),
                                   C.byref(aux), _ptr(total_out), _ptr(fixed_out), records.data_ptr(), max_det,
                                   _ptr(det), self._stream()))
        return records if det is None else (records, det)

    def _host_args(self, frames, samples, n_pairs, pair_stride, flow_out, fixed_out, records, fixed_packed=False,
                   stream_step=False):
        if n_pairs is None:
            n_pairs = frames.shape[0] - 1 if pair_stride == 1 else frames.shape[0] // 2
        if records is None:
            records = np.empty((n_pairs,), dtype=RECORD_DTYPE)
        for name, a in (('frames', frames), ('samples', samples), ('flow_out', flow_out), ('fixed_out', fixed_out)):
            if a is not None and not a.flags['C_CONTIGUOUS']:
                raise ValueError('%s must be C-contiguous' % name)
        if samples.dtype != np.int32 or samples.size < n_pairs * _lib.SAMPLES_PER_FRAME:
            raise ValueError('samples must be int32 (n, %d)' % _lib.SAMPLES_PER_FRAME)
        need = n_pairs if stream_step else n_pairs + 1 if pair_stride == 1 else 2 * n_pairs
        if frames is not None and (frames.dtype != np.uint8 or frames.shape[0] < need or
                                   tuple(frames.shape[1:]) not in ((self.height, self.width),
                                                                   (self.height, self.width, 3))):
            raise ValueError('frames must be uint8 (>=%d, %d, %d) gray or (>=%d, %d, %d, 3) BGR'
                             % (need, self.height, self.width, need, self.height, self.width))
        if fixed_out is not None:
            want = n_pairs * (self.packed_mask_bytes if fixed_packed else self.width * self.height)
            if fixed_out.dtype != np.uint8 or fixed_out.size < want:
                raise ValueError('fixed_out must be uint8 with at least %d elements' % want)
        return n_pairs, records

    def process_host(self, frames: np.ndarray, imu, samples: np.ndarray, n_pairs: Optional[int] = None,
                     pair_stride: int = 1, sky: Optional[np.ndarray] = None, seg: Optional[np.ndarray] = None,
                     flow_out: Optional[np.ndarray] = None, fixed_out: Optional[np.ndarray] = None,
                     records: Optional[np.ndarray] = None, **kw) -> np.ndarray:
        """The end-to-end call: HOST buffers in, HOST records (and optional masks / flow) out.  Frames may be gray
        (F, H, W) or BGR (F, H, W, 3).  Keyword options as in submit_host."""
        self.wait_host(0)
        records = self.submit_host(0, frames, imu, samples, n_pairs, pair_stride, sky, seg, flow_out, fixed_out,
                                   records, **kw)
        self.wait_host(0)
        return records

    def submit_host(self, slot: int, frames: np.ndarray, imu, samples: np.ndarray, n_pairs: Optional[int] = None,
                    pair_stride: int = 1, sky: Optional[np.ndarray] = None, seg: Optional[np.ndarray] = None,
                    flow_out: Optional[np.ndarray] = None, fixed_out: Optional[np.ndarray] = None,
                    records: Optional[np.ndarray] = None, gt_flow: Optional[np.ndarray] = None,
                    seg_packed: bool = False, sky_packed: bool = False, fixed_packed: bool = False,
                    copy_only: bool = False, detections: Optional[np.ndarray] = None) -> np.ndarray:
        """Asynchronous process_host: returns at once; the outputs are valid after wait_host(slot).  Keeping
        up to _lib.HOST_SLOTS batches in flight overlaps the host<->device copies with the compute.
        seg_packed / sky_packed: the masks are given at 1 bit per pixel (pack_mask_host); fixed_packed: fixed_out
        receives (n, packed_mask_bytes) bits; copy_only: move the bytes but skip the compute (host-feed ceiling);
        detections: an (n, max_det) DETECTION_DTYPE host array (pinned) that receives each pair's detection table."""
        return self._submit_host(slot, frames, None, imu, samples, n_pairs, pair_stride, sky, seg, flow_out, fixed_out,
                                 records, gt_flow, seg_packed, sky_packed, fixed_packed, copy_only, detections)

    def _submit_host(self, slot, frames, ids, imu, samples, n_pairs, pair_stride, sky, seg, flow_out, fixed_out, records,
                     gt_flow, seg_packed, sky_packed, fixed_packed, copy_only, detections) -> np.ndarray:
        """submit_host (ids None) or stream_submit_host."""
        if ids is not None:
            n_pairs, id_arr = self._stream_ids(ids)
        n_pairs, records = self._host_args(frames, samples, n_pairs, pair_stride, flow_out, fixed_out, records,
                                           fixed_packed, stream_step=ids is not None)
        aux = self._aux(sky, seg, gt_flow, n_pairs, host=True, sky_packed=sky_packed, seg_packed=seg_packed)
        flags = (_lib.HOST_BGR if frames.ndim == 4 else 0) | (_lib.HOST_SEG_PACKED if seg_packed else 0) | \
            (_lib.HOST_SKY_PACKED if sky_packed else 0) | (_lib.HOST_FIXED_PACKED if fixed_packed else 0) | \
            (_lib.HOST_COPY_ONLY if copy_only else 0)
        max_det, det = self._det_host(detections, n_pairs)
        if ids is None:
            if not copy_only:
                self.stream_epoch += 1
            check(self.lib.mavd_submit_host(self._h, slot, _hp(frames), n_pairs, pair_stride, imu,
                                            C.byref(self.detect_params), _hp(samples), C.byref(aux), flags,
                                            _hp(flow_out), _hp(fixed_out), records.ctypes.data, max_det, det,
                                            self._stream()))
        else:
            check(self.lib.mavd_stream_submit_host(self._h, slot, _hp(frames), n_pairs, id_arr, imu,
                                                   C.byref(self.detect_params), _hp(samples), C.byref(aux), flags,
                                                   _hp(flow_out), _hp(fixed_out), records.ctypes.data, max_det, det,
                                                   self._stream()))
        # keep the host buffers alive until the wait
        self._inflight[slot] = (frames, imu, samples, sky, seg, gt_flow, flow_out, fixed_out, records, detections)
        return records

    def wait_host(self, slot: int) -> None:
        check(self.lib.mavd_wait_host(self._h, slot))
        self._inflight.pop(slot, None)

    # -- frame streams (include/mavd.h: mavd_stream_start) ------------------------------------------
    def open_stream(self) -> int:
        """A free stream id of this engine (0 .. max_pairs-1).  Raises ValueError when all max_pairs are open."""
        for i in range(self.max_pairs):
            if i not in self._open_streams:
                self._open_streams.add(i)
                return i
        raise ValueError('all %d frame streams of this engine are open' % self.max_pairs)

    def close_stream(self, stream_id: int) -> None:
        """Give a stream id back to open_stream."""
        self._open_streams.discard(int(stream_id))

    def _stream_ids(self, ids: Iterable[int]) -> Tuple[int, C.Array]:
        ids = [int(i) for i in ids]
        return len(ids), (C.c_int32 * max(1, len(ids)))(*ids)

    def _check_stream_frames(self, frames: torch.Tensor, n: int) -> None:
        if frames.dtype != torch.uint8 or not frames.is_cuda or not frames.is_contiguous() or frames.dim() != 3 or \
                tuple(frames.shape) != (n, self.height, self.width):
            raise ValueError('frames must be a contiguous CUDA uint8 tensor (%d, %d, %d): one new frame per id'
                             % (n, self.height, self.width))

    def stream_start(self, frames: torch.Tensor, ids: Sequence[int]) -> None:
        """(Re)start the streams `ids` with frames[i] as stream ids[i]'s first frame (no flow)."""
        n, id_arr = self._stream_ids(ids)
        self._check_stream_frames(frames, n)
        check(self.lib.mavd_stream_start(self._h, frames.data_ptr(), n, id_arr, self._stream()))

    def stream_farneback(self, frames: torch.Tensor, ids: Sequence[int],
                         out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One step of the streams `ids`: flow of (stream ids[i]'s kept frame, frames[i]) for every i, which is then
        kept.  Equals farneback() with pair_stride 2 on the explicit pairs, bit for bit."""
        n, id_arr = self._stream_ids(ids)
        self._check_stream_frames(frames, n)
        if out is None:
            out = torch.empty((n, self.height, self.width, 2), dtype=torch.float32, device=self.device)
        check(self.lib.mavd_stream_farneback(self._h, frames.data_ptr(), n, id_arr, out.data_ptr(), self._stream()))
        return out

    def stream_process(self, frames: torch.Tensor, ids: Sequence[int], imu, samples: torch.Tensor,
                       sky: Optional[torch.Tensor] = None, seg: Optional[torch.Tensor] = None,
                       flow_out: Optional[torch.Tensor] = None, total_out: Optional[torch.Tensor] = None,
                       fixed_out: Optional[torch.Tensor] = None, records: Optional[torch.Tensor] = None,
                       gt_flow: Optional[torch.Tensor] = None, detections: Optional[int] = None):
        """process() for one step of the streams `ids` (stream_farneback's pairs); returns what process() returns."""
        n, id_arr = self._stream_ids(ids)
        self._check_stream_frames(frames, n)
        self._check_samples(samples, n)
        if records is None:
            records = torch.empty((n, RECORD_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        aux = self._aux(sky, seg, gt_flow, n)
        max_det, det = self._det_device(detections, n)
        check(self.lib.mavd_stream_process(self._h, frames.data_ptr(), n, id_arr, imu, C.byref(self.detect_params),
                                           samples.data_ptr(), C.byref(aux), _ptr(flow_out), _ptr(total_out),
                                           _ptr(fixed_out), records.data_ptr(), max_det, _ptr(det), self._stream()))
        return records if det is None else (records, det)

    def stream_submit_host(self, slot: int, frames: np.ndarray, ids: Sequence[int], imu, samples: np.ndarray,
                           sky: Optional[np.ndarray] = None, seg: Optional[np.ndarray] = None,
                           flow_out: Optional[np.ndarray] = None, fixed_out: Optional[np.ndarray] = None,
                           records: Optional[np.ndarray] = None, gt_flow: Optional[np.ndarray] = None,
                           seg_packed: bool = False, sky_packed: bool = False, fixed_packed: bool = False,
                           copy_only: bool = False, detections: Optional[np.ndarray] = None) -> np.ndarray:
        """submit_host for one step of the streams `ids`: HOST frames (n, H, W) gray or (n, H, W, 3) BGR, one per id;
        outputs valid after wait_host(slot)."""
        return self._submit_host(slot, frames, ids, imu, samples, None, 2, sky, seg, flow_out, fixed_out, records,
                                 gt_flow, seg_packed, sky_packed, fixed_packed, copy_only, detections)

    def detect_host(self, flow: np.ndarray, imu, samples: np.ndarray, sky: Optional[np.ndarray] = None,
                    seg: Optional[np.ndarray] = None, fixed_out: Optional[np.ndarray] = None,
                    records: Optional[np.ndarray] = None, gt_flow: Optional[np.ndarray] = None,
                    seg_packed: bool = False, sky_packed: bool = False, fixed_packed: bool = False,
                    detections: Optional[np.ndarray] = None) -> np.ndarray:
        """Detection from a HOST float32 flow (n, H, W, 2): what Processor.run_detection does with
        Dataset.get_flow_uv (processor.py:305-362).  detections: as in submit_host."""
        if flow.dtype != np.float32 or tuple(flow.shape[1:]) != (self.height, self.width, 2) or \
                not flow.flags['C_CONTIGUOUS']:
            raise ValueError('flow must be C-contiguous float32 (n, %d, %d, 2)' % (self.height, self.width))
        n, records = self._host_args(None, samples, flow.shape[0], 1, None, fixed_out, records, fixed_packed)
        aux = self._aux(sky, seg, gt_flow, n, host=True, sky_packed=sky_packed, seg_packed=seg_packed)
        flags = (_lib.HOST_SEG_PACKED if seg_packed else 0) | (_lib.HOST_SKY_PACKED if sky_packed else 0) | \
            (_lib.HOST_FIXED_PACKED if fixed_packed else 0)
        max_det, det = self._det_host(detections, n)
        check(self.lib.mavd_detect_host(self._h, flow.ctypes.data, n, imu, C.byref(self.detect_params), _hp(samples),
                                        C.byref(aux), flags, _hp(fixed_out), records.ctypes.data, max_det, det,
                                        self._stream()))
        return records

    @staticmethod
    def records_to_numpy(records: torch.Tensor) -> np.ndarray:
        return records.cpu().numpy().view(RECORD_DTYPE).reshape(-1)

    @staticmethod
    def stats_to_numpy(stats: torch.Tensor) -> np.ndarray:
        return stats.cpu().numpy().view(STATS_DTYPE).reshape(-1)

    def force_generic_iteration(self, on: bool = True) -> None:
        """Tests only: use the non-TMA iteration kernel even where the TMA kernel applies."""
        check(self.lib.mavd_debug_force_generic_iteration(self._h, 1 if on else 0))

    def force_exact_residual(self, on: bool = True) -> None:
        """Tests only: evaluate every pixel of the residual stage in float64 (no float32 pre-decision)."""
        check(self.lib.mavd_debug_force_exact_residual(self._h, 1 if on else 0))

    def profile_enable(self, on: bool = True) -> None:
        check(self.lib.mavd_profile_enable(self._h, 1 if on else 0))

    def profile_read(self) -> Dict[str, Tuple[float, int]]:
        """{kernel class: (summed device ms, timed launch groups)} since profile_enable()."""
        prof = _lib.Profile()
        check(self.lib.mavd_profile_read(self._h, C.byref(prof)))
        return {n: (prof.ms[i], int(prof.launches[i])) for i, n in enumerate(_lib.PROF_NAMES)}

    def profile_timeline(self, max_records: int = 4096):
        """[(kernel class, start ms, end ms)] of every timed launch group since profile_enable(), in launch order."""
        buf = (C.c_double * (3 * max_records))()
        n = C.c_int32()
        check(self.lib.mavd_profile_timeline(self._h, buf, max_records, C.byref(n)))
        names = _lib.PROF_NAMES
        return [(names[int(buf[3 * i])] if int(buf[3 * i]) < len(names) else str(int(buf[3 * i])), buf[3 * i + 1],
                 buf[3 * i + 2]) for i in range(n.value)]

    def launch_count(self) -> int:
        return int(self.lib.mavd_launch_count())

    def graph_stats(self) -> Dict[str, int]:
        """Launch sequences held by the handle: replayed as CUDA graphs / run kernel by kernel (capture failed)."""
        a, b = C.c_int32(), C.c_int32()
        check(self.lib.mavd_graph_stats(self._h, C.byref(a), C.byref(b)))
        return {'captured': a.value, 'direct': b.value}


_SHARED: Dict[tuple, 'Engine'] = {}


def shared_engine(width: int, height: int, params: Optional[Dict] = None, max_pairs: int = 1,
                  device: Optional[int] = None) -> 'Engine':
    """One cached Engine per (device, W, H, Farneback parameters, max_pairs) for the reference-named classes
    (Farneback, Detector, FocusOfExpansion, Processor), which all work on the same frame geometry."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    p = dict(REFERENCE_PARAMS)
    if params:
        p.update(params)
    key = (device, int(width), int(height), int(max_pairs), tuple(sorted(p.items())))
    eng = _SHARED.get(key)
    if eng is None or not eng._h.value:
        eng = Engine(width, height, p, max_pairs=max_pairs, device=device)
        _SHARED[key] = eng
    return eng
