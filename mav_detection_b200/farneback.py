"""Farneback with the reference's API (/root/reference/src/farneback.py:12-107) on the CUDA path.

    Farneback(capture, output).process() -> (H, W, 3) uint8 BGR visualisation

`capture` is anything with cv2.VideoCapture's `read() -> (ok, BGR frame)`.  process() reads the next frame,
converts it to gray on the device (mavd_bgr2gray == cv2.cvtColor, :74), computes the dense flow against the
previous frame with the reference's parameters (mavd_farneback == cv2.calcOpticalFlowFarneback(..., 0.4, 1, 12,
10, 8, 1.2, 0), :76-80), keeps `prevgray` (:81) and returns the HSV visualisation (:83-99) built by
mavd_flow_vis.  The previous frame is kept expanded on the device in one frame stream of the engine
(mavd_stream_farneback), so each call expands only the new frame; when the engine has no free stream the call pairs
the two frames explicitly, with the same result.  Another user's non-stream call on the engine ends the stream; after
that has happened before two calls in a row, process() pairs explicitly (one launch sequence, where a restart and a
step would take two) until a call finds that nobody else used the engine since the previous one.  The reference discards the flow; here it stays available as `self.flow` ((H, W, 2) float32
CUDA tensor) for callers that want the field itself.  draw_flow / draw_hsv / warp_flow (:28-69) are unused
drawing helpers and are not rebuilt."""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Any, Dict, Optional

import numpy as np

from . import _lib
from ._lib import check

# src/farneback.py:78-80
PROCESS_PARAMS: Dict[str, Any] = dict(pyr_scale=0.4, levels=1, winsize=12, iterations=10, poly_n=8, poly_sigma=1.2,
                                      flags=0)


class Farneback:
    def __init__(self, capture: Any, output: Any = None, engine: Any = None) -> None:
        import torch
        self.capture = capture
        self.output = output
        _, prev = self.capture.read()
        prev = np.ascontiguousarray(prev)
        if prev.ndim != 3 or prev.shape[2] != 3 or prev.dtype != np.uint8:
            raise ValueError('Farneback expects (H, W, 3) uint8 BGR frames')
        capture_size = prev.shape
        if engine is None:
            from . import engine as engine_mod
            engine = engine_mod.shared_engine(prev.shape[1], prev.shape[0], PROCESS_PARAMS, max_pairs=1)
        self._eng = engine
        self._torch = torch
        self.hsv = np.zeros_like(prev)
        self._prevgray_d = engine.bgr2gray(torch.from_numpy(prev).to(engine.device))
        self.cur_glitch = prev.copy()
        self.history_length = 1
        self.prev_results = np.zeros((*capture_size, self.history_length))
        self.rolling_history_id = 0
        self.flow: Optional['torch.Tensor'] = None
        self._scratch = torch.zeros((3,), dtype=torch.int32, device=engine.device)
        self._live = False               # the stream holds prevgray
        self._ended_in_a_row = 0         # calls in a row before which another user's non-stream call ended the stream
        self._stream_epoch = engine.stream_epoch
        try:
            self._stream: Optional[int] = engine.open_stream()
        except ValueError:
            self._stream = None          # every stream of the engine is taken: explicit pairs
        else:
            weakref.finalize(self, engine.close_stream, self._stream)

    @property
    def prevgray(self) -> np.ndarray:
        return self._prevgray_d.cpu().numpy()

    def process(self) -> np.ndarray:
        torch, eng = self._torch, self._eng
        _, img = self.capture.read()
        img = np.ascontiguousarray(img)
        gray = eng.bgr2gray(torch.from_numpy(img).to(eng.device))
        # a non-stream Farneback call by another user of the engine since our last call ended the stream
        ended = eng.stream_epoch != self._stream_epoch
        self._ended_in_a_row = self._ended_in_a_row + 1 if ended else 0
        if self._stream is None or self._ended_in_a_row >= 2:
            self.flow = eng.farneback(torch.stack([self._prevgray_d, gray]), n_pairs=1)[0]
            self._live = False           # that call ended our stream too
        else:
            if ended or not self._live:
                eng.stream_start(self._prevgray_d[None], [self._stream])
            self.flow = eng.stream_farneback(gray[None], [self._stream])[0]
            self._live = True
        self._stream_epoch = eng.stream_epoch
        self._prevgray_d = gray
        h, w = gray.shape
        bgr = torch.empty((h, w, 3), dtype=torch.uint8, device=eng.device)
        with torch.cuda.device(eng.device):      # handle-less entry point: runs on the current device
            check(eng.lib.mavd_flow_vis(self.flow.data_ptr(), h * w, bgr.data_ptr(), self._scratch.data_ptr(),
                                        torch.cuda.current_stream(eng.device).cuda_stream))
        nonzero_values = int(self._scratch[2].item()) & 0xffffffff
        invalid_frame = nonzero_values < 1
        result = bgr.cpu().numpy()
        if invalid_frame:
            result = self.prev_results[..., 0].astype(np.uint8)
        self.prev_results[..., self.rolling_history_id] = result
        if self.rolling_history_id >= self.history_length:
            self.rolling_history_id = 0
        return result
