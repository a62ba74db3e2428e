"""bench.py --dump-outputs: the files it writes (CPU) and that two runs with the same arguments agree (GPU)."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _records(n):
    from mav_detection_b200.engine import RECORD_DTYPE
    rec = np.zeros((n,), RECORD_DTYPE)
    rng = np.random.default_rng(3)
    rec['foe'] = rng.random((n, 2)) * 1000
    rec['n_labels'] = np.arange(n) + 7
    rec['stats']['n_fixed'] = 2 ** 40 + np.arange(n)
    rec['stats']['seg_bbox'] = rng.integers(-1, 1000, (n, 4))
    rec['boxes'] = rng.integers(0, 2 ** 21, (n, 32, 5))
    return rec


def _load(d):
    return {os.path.basename(p)[:-4]: np.load(p) for p in sorted(glob.glob(os.path.join(d, '*.npy')))}


def test_dump_writes_every_record_field_and_the_whole_small_mask(tmp_path):
    import bench
    rec = _records(3)
    fixed = (np.random.default_rng(4).random((3, 8, 10)) < 0.3).astype(np.uint8)
    bench.dump_outputs(str(tmp_path / 'out'), rec, fixed)
    got = _load(str(tmp_path / 'out'))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got['fixed'], fixed) and got['fixed'].dtype == np.float32
    assert np.array_equal(got['records_foe'], rec['foe'])
    assert np.array_equal(got['records_n_labels'], rec['n_labels'])
    assert np.array_equal(got['records_stats_n_fixed'], rec['stats']['n_fixed'])
    assert np.array_equal(got['records_stats_seg_bbox'], rec['stats']['seg_bbox'])
    assert np.array_equal(got['records_boxes'], rec['boxes'])
    for sub in rec.dtype['stats'].names:
        assert 'records_stats_' + sub in got


def test_dump_of_a_c2_step_is_a_fixed_sample_under_64_mb(tmp_path):
    import bench
    W, H, _, B, _, _ = bench.WORKLOADS['c2']
    fixed = np.zeros((B, H, W), np.uint8)
    fixed[:, ::7, ::3] = 1
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), _records(B), fixed)
    a, b = _load(str(tmp_path / 'a')), _load(str(tmp_path / 'b'))
    assert sorted(a) == sorted(b) and 'fixed' not in a
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    idx = a['fixed_sample_index'].astype(np.int64)
    assert idx.size > bench.DUMP_MASK_SAMPLES * 0.9 and np.all(np.diff(idx) > 0) and idx[-1] < fixed.size
    assert np.array_equal(a['fixed_sample'], fixed.reshape(-1)[idx])
    total = sum(os.path.getsize(p) for p in glob.glob(str(tmp_path / 'a' / '*.npy')))
    assert total <= 64 << 20, total


@pytest.mark.gpu
def test_two_runs_dump_the_same_outputs(tmp_path):
    """Same arguments, same outputs: every dumped array is bit-identical between two runs, except the segmentation
    flow sums, which the residual kernel accumulates with double-precision atomics in no fixed order."""
    outs = []
    for d in ('a', 'b'):
        res = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'c3', '--pairs', '4',
                              '--steps', '3', '--warmup', '3', '--no-cpu', '--dump-outputs', str(tmp_path / d)],
                             cwd=ROOT, capture_output=True, text=True)
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line['steps'] == 3 and line['config']['pairs_per_step'] == 4
        outs.append(_load(str(tmp_path / d)))
    a, b = outs
    assert sorted(a) == sorted(b)
    assert a['fixed'].shape == (4, 480, 640) and a['records_foe'].shape == (4, 2)
    assert a['fixed'].sum() == a['records_stats_n_fixed'].sum()
    for k in a:
        if k == 'records_stats_seg_flow_sum':
            assert np.allclose(a[k], b[k], rtol=1e-12, atol=1e-9), k
        else:
            assert np.array_equal(a[k], b[k]), k
