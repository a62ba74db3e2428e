"""ctypes binding of libmavd.so (include/mavd.h).  There is no CPU fallback: if the CUDA library
has not been built, importing a compute entry point raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libmavd.so')

ABI_VERSION = 3
MAVD_OK, MAVD_ERR_INVALID, MAVD_ERR_CUDA, MAVD_ERR_UNSUPPORTED, MAVD_ERR_NOMEM = 0, 1, 2, 3, 4
N_SAMPLE_PAIRS = 1000
SAMPLES_PER_FRAME = 4 * N_SAMPLE_PAIRS
MAX_BOXES = 32
HOST_SLOTS = 3
MAX_DETECTIONS = 256
OPTFLOW_FARNEBACK_GAUSSIAN = 256
LK_GET_MIN_EIGENVALS = 8
LK_MAX_LEVEL = 16
TERM_COUNT, TERM_EPS = 1, 2


class FarnebackParams(C.Structure):
    _fields_ = [('pyr_scale', C.c_double), ('levels', C.c_int32), ('winsize', C.c_int32),
                ('iterations', C.c_int32), ('poly_n', C.c_int32), ('poly_sigma', C.c_double),
                ('flags', C.c_int32)]


class Config(C.Structure):
    _fields_ = [('device', C.c_int32), ('width', C.c_int32), ('height', C.c_int32),
                ('max_pairs', C.c_int32), ('farneback', FarnebackParams)]


class Imu(C.Structure):
    _fields_ = [('ang', C.c_double * 3), ('dt', C.c_double), ('derotate', C.c_int32), ('_pad', C.c_int32)]


class DetectParams(C.Structure):
    _fields_ = [('magnitude_threshold', C.c_double), ('ransac_threshold', C.c_double),
                ('dyn_offset', C.c_double), ('dyn_base', C.c_double), ('dyn_gain', C.c_double),
                ('dyn_min_mag', C.c_double), ('fixed_min_mag', C.c_double), ('fixed_angle', C.c_double)]


class FrameStats(C.Structure):
    _fields_ = [('max_phi', C.c_double), ('n_total', C.c_int64), ('n_fixed', C.c_int64),
                ('positives', C.c_int64), ('negatives', C.c_int64), ('tp_total', C.c_int64),
                ('fp_total', C.c_int64), ('tp_fixed', C.c_int64), ('fp_fixed', C.c_int64),
                ('seg_bbox', C.c_int32 * 4), ('seg_flow_sum', C.c_double * 2), ('gt_flow_sum', C.c_double * 2)]


class FrameRecord(C.Structure):
    _fields_ = [('foe', C.c_double * 2), ('n_intersections', C.c_int32), ('n_labels', C.c_int32),
                ('stats', FrameStats), ('boxes', (C.c_int32 * 5) * MAX_BOXES)]


class Detection(C.Structure):
    """One entry of a frame's detection table (include/mavd.h: mavd_detection)."""
    _fields_ = [('label', C.c_int32), ('box', C.c_int32 * 4), ('area', C.c_int32), ('sum_x', C.c_int64),
                ('sum_y', C.c_int64), ('flow_sum', C.c_double * 2)]


class GfttParams(C.Structure):
    """Arguments of cv2.goodFeaturesToTrack (include/mavd.h: mavd_gftt_params)."""
    _fields_ = [('max_corners', C.c_int32), ('quality_level', C.c_double), ('min_distance', C.c_double),
                ('block_size', C.c_int32), ('gradient_size', C.c_int32)]


class LkParams(C.Structure):
    """Arguments of cv2.calcOpticalFlowPyrLK (include/mavd.h: mavd_lk_params)."""
    _fields_ = [('win_w', C.c_int32), ('win_h', C.c_int32), ('max_level', C.c_int32), ('criteria_type', C.c_int32),
                ('criteria_count', C.c_int32), ('criteria_eps', C.c_double), ('flags', C.c_int32),
                ('min_eig_threshold', C.c_double)]


class Tuning(C.Structure):
    """Launch-shape choices (include/mavd.h: mavd_tuning); results never depend on them."""
    _fields_ = [('mat_coord', C.c_int32), ('pyr_staged', C.c_int32), ('use_graph', C.c_int32),
                ('polyexp_tma', C.c_int32), ('iter_small_tiles', C.c_int32), ('use_pdl', C.c_int32),
                ('pyr_sweep', C.c_int32), ('reserved', C.c_int32 * 1)]


class AuxInputs(C.Structure):
    """Optional per-frame inputs of the detection stages (include/mavd.h: mavd_aux_inputs)."""
    _fields_ = [('sky', C.c_void_p), ('sky_stride', C.c_int64), ('seg', C.c_void_p), ('seg_stride', C.c_int64),
                ('gt_flow', C.c_void_p)]


HOST_BGR, HOST_SEG_PACKED, HOST_SKY_PACKED, HOST_FIXED_PACKED, HOST_COPY_ONLY = 1, 2, 4, 8, 16

PROF_CLASSES = 12
PROF_NAMES = ['pyramid', 'polyexp', 'matrices', 'iter_full', 'iter_full_last', 'iter_coarse', 'foe', 'residual',
              'ccl']


class Profile(C.Structure):
    _fields_ = [('ms', C.c_double * PROF_CLASSES), ('launches', C.c_int64 * PROF_CLASSES)]


# every symbol include/mavd.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    'mavd_abi_version': (C.c_int, []),
    'mavd_last_error': (C.c_char_p, []),
    'mavd_default_detect_params': (None, [C.POINTER(DetectParams)]),
    'mavd_create': (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    'mavd_destroy': (C.c_int, [_P]),
    'mavd_workspace_bytes': (C.c_int, [_P, C.POINTER(C.c_size_t)]),
    'mavd_default_tuning': (None, [C.POINTER(Tuning)]),
    'mavd_set_tuning': (C.c_int, [_P, C.POINTER(Tuning)]),
    'mavd_get_tuning': (C.c_int, [_P, C.POINTER(Tuning)]),
    'mavd_level_info': (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'mavd_bgr2gray': (C.c_int, [_P, _P, C.c_int64, _P]),
    'mavd_farneback': (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    'mavd_farneback_tap': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    'mavd_derotate': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), _P, _P]),
    'mavd_derotate_f64': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), _P, _P]),
    'mavd_foe': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P, _P, _P, _P]),
    'mavd_foe_dense': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(DetectParams), _P, _P, _P, _P]),
    'mavd_ransac': (C.c_int, [_P, _P, C.c_int32, C.c_double, _P, _P]),
    'mavd_get_phi': (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    'mavd_residual_masks': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                      _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P, _P]),
    'mavd_ccl': (C.c_int, [_P, _P, C.c_int32, _P, _P, C.c_int32, _P, _P]),
    'mavd_process': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                               _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P, _P]),
    'mavd_process_host': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                    _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P]),
    'mavd_detect': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P, _P, C.c_int64, _P, C.c_int64,
                              _P, _P, _P, _P]),
    'mavd_submit_host': (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                   _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P]),
    'mavd_submit_host_bgr': (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                       _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P]),
    'mavd_wait_host': (C.c_int, [_P, C.c_int32]),
    'mavd_detect_host': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P, _P, C.c_int64, _P,
                                   C.c_int64, _P, _P, _P]),
    'mavd_detect_ex': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P, C.POINTER(AuxInputs),
                                 _P, _P, _P, _P]),
    'mavd_process_ex': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                  C.POINTER(AuxInputs), _P, _P, _P, _P, _P]),
    'mavd_submit_host_ex': (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams),
                                      _P, C.POINTER(AuxInputs), C.c_int32, _P, _P, _P, _P]),
    'mavd_detect_host_ex': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                      C.POINTER(AuxInputs), C.c_int32, _P, _P, _P]),
    'mavd_detections': (C.c_int, [_P, _P, C.c_int32, _P, C.POINTER(Imu), C.c_int32, _P, _P]),
    'mavd_detect_det': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P, C.POINTER(AuxInputs),
                                  _P, _P, _P, C.c_int32, _P, _P]),
    'mavd_process_det': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                   C.POINTER(AuxInputs), _P, _P, _P, _P, C.c_int32, _P, _P]),
    'mavd_submit_host_det': (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams),
                                       _P, C.POINTER(AuxInputs), C.c_int32, _P, _P, _P, C.c_int32, _P, _P]),
    'mavd_detect_host_det': (C.c_int, [_P, _P, C.c_int32, C.POINTER(Imu), C.POINTER(DetectParams), _P,
                                       C.POINTER(AuxInputs), C.c_int32, _P, _P, C.c_int32, _P, _P]),
    'mavd_good_features_to_track': (C.c_int, [_P, _P, C.c_int32, C.POINTER(GfttParams), _P, C.c_int64, _P, _P, _P,
                                               _P]),
    'mavd_pyr_lk': (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(LkParams), _P, C.c_int32, _P, _P, _P, _P, _P]),
    'mavd_packed_mask_bytes': (C.c_int64, [C.c_int32, C.c_int32]),
    'mavd_pack_mask': (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P]),
    'mavd_unpack_mask': (C.c_int, [_P, C.c_int32, C.c_int64, C.c_uint8, _P, _P]),
    'mavd_magnitude': (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P]),
    'mavd_simple_bbox': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    'mavd_tpr_fpr_counts': (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    'mavd_flow_vis': (C.c_int, [_P, C.c_int64, _P, _P, _P]),
    'mavd_phi_colormap': (C.c_int, [_P, C.c_int32, C.c_int64, C.c_double, _P, _P, _P]),
    'mavd_mask_overlay': (C.c_int, [_P, C.c_int32, _P, C.c_int64, _P, _P, _P]),
    'mavd_launch_count': (C.c_int64, []),
    'mavd_graph_stats': (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'mavd_debug_force_generic_iteration': (C.c_int, [_P, C.c_int32]),
    'mavd_debug_force_exact_residual': (C.c_int, [_P, C.c_int32]),
    'mavd_profile_enable': (C.c_int, [_P, C.c_int32]),
    'mavd_profile_read': (C.c_int, [_P, C.POINTER(Profile)]),
    'mavd_profile_timeline': (C.c_int, [_P, C.POINTER(C.c_double), C.c_int32, C.POINTER(C.c_int32)]),
}

_lib: Optional[C.CDLL] = None


class MavdError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libmavd.so.  Raises (never falls back) when the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MavdError('libmavd.so is not built (%s). Run `python -c "import __graft_entry__ as g; g.build()"` '
                        'from the repository root; there is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    assert lib.mavd_abi_version() == ABI_VERSION
    _lib = lib
    return lib


def check(status: int) -> None:
    """Map the C status to the exception type the reference would raise (SURVEY §8b: errors)."""
    if status == MAVD_OK:
        return
    msg = load().mavd_last_error().decode('utf-8', 'replace')
    if status in (MAVD_ERR_INVALID, MAVD_ERR_UNSUPPORTED):
        raise ValueError(msg)
    if status == MAVD_ERR_NOMEM:
        raise MemoryError(msg)
    raise MavdError(msg)
