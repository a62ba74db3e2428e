"""CPU: the C-ABI library loads and exports every symbol include/mavd.h declares; struct layouts agree."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    from mav_detection_b200 import _lib, build
    build.build()
    return _lib.load()


def _declared_functions():
    src = open(os.path.join(ROOT, 'include', 'mavd.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(mavd_[a-z0-9_]+)\s*\(', src)))


def test_every_declared_symbol_is_exported_and_bound(lib):
    from mav_detection_b200 import _lib
    names = _declared_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), 'libmavd.so does not export %s' % n
        assert n in _lib.SIGNATURES, '%s has no ctypes signature' % n
    assert sorted(_lib.SIGNATURES) == names


def test_ctypes_signatures_have_the_header_arity_and_return_types():
    """A binding that drifts from include/mavd.h corrupts the call silently: every prototype's parameter count and
    return type (int status / int64 counter / const char*) must be what mav_detection_b200/_lib.py declares."""
    from mav_detection_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'mavd.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    src = re.sub(r'//[^\n]*', '', src)
    decls = re.findall(r'\b(int64_t|int|void|const char\*)\s+(mavd_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;', src, flags=re.S)
    assert sorted(d[1] for d in decls) == _declared_functions()
    restype = {'int': C.c_int, 'int64_t': C.c_int64, 'const char*': C.c_char_p, 'void': None}
    for ret, name, args in decls:
        args = args.strip()
        n = 0 if args in ('', 'void') else len(args.split(','))
        res, argtypes = _lib.SIGNATURES[name]
        assert len(argtypes) == n, '%s: header has %d parameters, ctypes %d' % (name, n, len(argtypes))
        assert res is restype[ret], '%s: header returns %s' % (name, ret)


def test_abi_version_4_and_defaults(lib):
    from mav_detection_b200 import _lib
    assert lib.mavd_abi_version() == _lib.ABI_VERSION == 4
    p = _lib.DetectParams()
    lib.mavd_default_detect_params(C.byref(p))
    # focus_of_expansion.py:22-23, processor.py:333-341
    assert (p.magnitude_threshold, p.ransac_threshold) == (2.5, 30.0)
    assert (p.dyn_offset, p.dyn_base, p.dyn_gain, p.dyn_min_mag, p.fixed_min_mag, p.fixed_angle) == \
        (0.25, 0.5, 8.0, 0.5, 1.0, 15.0)


def test_struct_layouts_of_abi_4():
    from mav_detection_b200 import _lib
    assert C.sizeof(_lib.Imu) == 40
    assert C.sizeof(_lib.FarnebackParams) == 40
    assert C.sizeof(_lib.FrameStats) == 8 * 9 + 16 + 16 + 16
    assert C.sizeof(_lib.Tuning) == 8 * 4 and C.sizeof(_lib.AuxInputs) == 40
    assert C.sizeof(_lib.FrameRecord) == 16 + 8 + C.sizeof(_lib.FrameStats) + 32 * 5 * 4
    assert np.dtype(_lib.FrameRecord).itemsize == C.sizeof(_lib.FrameRecord)


def test_tuning_fields_are_the_header_members():
    """The ctypes Tuning fields are the mavd_tuning members of include/mavd.h by name, order and array length: a list
    that drifts from the header can keep the struct's size and then sets the wrong switch without an error."""
    from mav_detection_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'mavd.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    body = re.search(r'typedef struct mavd_tuning \{(.*?)\} mavd_tuning;', src, flags=re.S).group(1)
    members = re.findall(r'int32_t\s+(\w+)(?:\[(\d+)\])?\s*;', body)
    assert [(n, int(k or 1)) for n, k in members] == \
        [(f, getattr(t, '_length_', 1)) for f, t in _lib.Tuning._fields_]
    assert len(members) == len(re.findall(r';', body))


def test_invalid_config_is_a_value_error_without_touching_the_gpu(lib):
    from mav_detection_b200 import _lib
    cfg = _lib.Config(0, 640, 480, 1, _lib.FarnebackParams(1.5, 1, 12, 10, 8, 1.2, 0))   # pyr_scale >= 1
    h = C.c_void_p()
    rc = lib.mavd_create(C.byref(cfg), C.byref(h))
    assert rc == _lib.MAVD_ERR_INVALID
    with pytest.raises(ValueError):
        _lib.check(rc)
    cfg = _lib.Config(0, 640, 480, 1, _lib.FarnebackParams(0.5, 1, 12, 10, 9, 1.2, 0))    # poly_n > 8
    assert lib.mavd_create(C.byref(cfg), C.byref(h)) == _lib.MAVD_ERR_UNSUPPORTED


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from mav_detection_b200 import _lib, engine
    with pytest.raises(_lib.MavdError):
        engine.Engine(64, 64)
