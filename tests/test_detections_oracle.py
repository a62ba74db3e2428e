"""CPU: the detection-table struct of the C ABI and its NumPy oracle (tests/detections_np.py).

The ctypes Detection must be include/mavd.h's mavd_detection member for member: a binding that drifts keeps a plausible
size and then reads the wrong bytes.  The oracle's boxes, areas and centroids must be cv2.connectedComponentsWithStats'
(8-connectivity), its order (area descending, then canonical label ascending) must be total, also when many
components have the same area."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import detections_np as dnp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_CTYPES = {'int32_t': C.c_int32, 'int64_t': C.c_int64, 'double': C.c_double}


def test_detection_struct_is_the_header_member_list():
    from mav_detection_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'mavd.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    body = re.search(r'typedef struct mavd_detection \{(.*?)\} mavd_detection;', src, flags=re.S).group(1)
    members = []
    for typ, names in re.findall(r'(int32_t|int64_t|double)\s+([^;]+);', body):
        for nm in names.split(','):
            m = re.fullmatch(r'\s*(\w+)(?:\[(\d+)\])?\s*', nm)
            members.append((m.group(1), _CTYPES[typ], int(m.group(2) or 1)))
    assert len(members) == 6
    fields = _lib.Detection._fields_
    assert [n for n, _, _ in members] == [f for f, _ in fields]
    offset = 0
    for (name, ctype, count), (fname, ftype) in zip(members, fields):
        base = getattr(ftype, '_type_', ftype) if hasattr(ftype, '_length_') else ftype
        assert base is ctype and getattr(ftype, '_length_', 1) == count, name
        offset = -(-offset // C.sizeof(ctype)) * C.sizeof(ctype)        # natural alignment, as the C compiler lays it
        assert getattr(_lib.Detection, name).offset == offset, name
        offset += C.sizeof(ctype) * count
    assert C.sizeof(_lib.Detection) == offset == 56
    assert _lib.MAX_DETECTIONS == int(re.search(r'#define MAVD_MAX_DETECTIONS (\d+)', src).group(1)) == 256
    from mav_detection_b200 import engine
    assert engine.DETECTION_DTYPE.itemsize == 56
    assert [engine.DETECTION_DTYPE.fields[n][1] for n in dnp.DETECTION_DTYPE.names] == \
        [dnp.DETECTION_DTYPE.fields[n][1] for n in dnp.DETECTION_DTYPE.names]


def _masks():
    rng = np.random.default_rng(11)
    out = []
    for h, w in ((8, 8), (17, 33), (64, 48), (120, 160)):
        for p in (0.05, 0.3, 0.5):
            out.append(('noise%g_%dx%d' % (p, w, h), (rng.random((h, w)) < p).astype(np.uint8)))
    # equal-area blobs: 2 x 2 squares on a 3-pixel grid, a few 1 x 4 bars of the same area among them
    m = np.zeros((60, 90), np.uint8)
    for y in range(0, 57, 3):
        for x in range(0, 87, 3):
            m[y:y + 2, x:x + 2] = 1
    m[0:1, 0:5] = 0
    m[0, 0:4] = 1
    out.append(('equal_area', m))
    iso = np.zeros((31, 41), np.uint8)
    iso[::2, ::2] = 1
    out.append(('isolated', iso))
    out.append(('empty', np.zeros((8, 8), np.uint8)))
    out.append(('full', np.ones((9, 13), np.uint8)))
    return out


@pytest.mark.parametrize('name,mask', _masks(), ids=[n for n, _ in _masks()])
@pytest.mark.parametrize('max_det', [1, 7, 32, 256])
def test_oracle_agrees_with_cv2(name, mask, max_det):
    cv2 = pytest.importorskip('cv2')
    from oracle import ccl_np
    n, lab, st, cen = cv2.connectedComponentsWithStats(mask, connectivity=8, ltype=cv2.CV_32S)
    # cv2 numbers components in its own order: map them to canonical labels by their first raster pixel
    canon = ccl_np.canonicalise(lab)
    cv_of = np.zeros(n, np.int64)
    cv_of[canon[lab > 0]] = lab[lab > 0]
    det = dnp.detections(mask, max_det=max_det)
    k = min(n - 1, max_det)
    assert np.all(det['label'][k:] == 0) and np.all(det['area'][k:] == 0) and np.all(det['box'][k:] == 0)
    rows = det[:k]
    c = cv_of[rows['label']]
    assert np.array_equal(rows['box'], st[c, :4])
    assert np.array_equal(rows['area'], st[c, 4])
    assert np.array_equal(rows['sum_x'] / rows['area'], cen[c, 0])
    assert np.array_equal(rows['sum_y'] / rows['area'], cen[c, 1])
    # the order: area descending, label ascending within an area, and nothing left out above the cut
    key = [(-a, l) for a, l in zip(rows['area'], rows['label'])]
    assert key == sorted(key)
    if n - 1 > k:
        rest = sorted((-st[cv_of[l], 4], l) for l in range(1, n) if l not in set(rows['label'].tolist()))
        assert rest[0] > key[-1]


def test_oracle_flow_sums_are_np_add_at():
    rng = np.random.default_rng(2)
    mask = (rng.random((40, 50)) < 0.4).astype(np.uint8)
    flow = rng.standard_normal((40, 50, 2))
    det = dnp.detections(mask, flow, max_det=256)
    from oracle import ccl_np
    lab, _ = ccl_np.label(mask)
    for d in det[det['label'] > 0]:
        sel = lab == d['label']
        assert np.allclose(d['flow_sum'], flow[sel].sum(axis=0), rtol=0, atol=1e-12)
    assert np.all(dnp.detections(mask, None, max_det=8)['flow_sum'] == 0)
