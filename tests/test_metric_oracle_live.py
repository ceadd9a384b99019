"""oracle/metric_oracle.py against the UNMODIFIED reference function ts_diff_metric
(train/scripts/stage2/stage2_metrics.py:22-88), compiled live from where it lies (the module itself imports pandas,
the sampler package and the training utilities at import time; only the one function is executed).  Skipped where
/root/reference is not mounted."""
import ast
import logging
import os

import numpy as np
import pytest

from oracle import metric_oracle as mo, ref_harness

pytestmark = pytest.mark.skipif(not ref_harness.available(), reason='/root/reference is not mounted')

EVENT_DTYPE = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])


def _reference_fn():
    path = os.path.join(ref_harness.REF_ROOT, 'train', 'scripts', 'stage2', 'stage2_metrics.py')
    tree = ast.parse(open(path).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == 'ts_diff_metric'][0]
    ns = {'np': np, 'logger': logging.getLogger('ref_metric')}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, 'exec'), ns)
    return ns['ts_diff_metric']


def _events(n, seed, spread, neg_polarity=False, box=((100, 112), (50, 60))):
    rng = np.random.default_rng(seed)
    ev = np.zeros(n, dtype=EVENT_DTYPE)
    ev['timestamp'] = rng.integers(0, spread, n)
    ev['x'] = rng.integers(*box[0], n)
    ev['y'] = rng.integers(*box[1], n)
    ev['polarity'] = rng.integers(0, 2, n)
    if neg_polarity:
        ev['polarity'][ev['polarity'] == 0] = -1
    return ev


@pytest.mark.parametrize('search_range,fps', [(0, 30), (1, 30), (2, 60)])
def test_metric_oracle_equals_reference(search_range, fps):
    ref = _reference_fn()
    gt = _events(300, 1, 40000, neg_polarity=True)
    pred = _events(260, 2, 40000)
    want = ref(gt.copy(), pred.copy(), search_range=search_range, fps=fps)
    got = mo.ts_diff_metric_oracle(gt, pred, search_range=search_range, fps=fps)
    assert got[1] == want[1] and got[1] > 0
    assert abs(got[0] - want[0]) <= 1e-9 * abs(want[0])


def _compare(gt, pred, search_range, fps):
    want = _reference_fn()(gt.copy(), pred.copy(), search_range=search_range, fps=fps)
    got = mo.ts_diff_metric_oracle(gt, pred, search_range=search_range, fps=fps)
    assert got[1] == want[1]
    assert abs(got[0] - want[0]) <= 1e-9 * max(abs(want[0]), 1.0)


@pytest.mark.parametrize('search_range,fps', [(0, 0.25), (1, 0.25), (5, 30)])
def test_metric_oracle_equals_reference_low_fps_wide_window(search_range, fps):
    """fps 0.25: the cap (1.2e6) exceeds the 1e6 a ground-truth event with no predicted event nearby adds; r = 5."""
    gt = _events(300, 3, 4 * 10 ** 6, neg_polarity=True)
    pred = _events(200, 4, 4 * 10 ** 6)
    _compare(gt, pred, search_range, fps)


@pytest.mark.parametrize('corner', [(0, 0), (342, 0), (0, 256), (342, 256)])
def test_metric_oracle_equals_reference_sensor_edges(corner):
    """Events in the 4x4 corners of the 346x260 sensor, where the window is clamped."""
    box = ((corner[0], corner[0] + 4), (corner[1], corner[1] + 4))
    gt = _events(200, 5, 40000, neg_polarity=True, box=box)
    pred = _events(150, 6, 40000, box=box)
    for search_range in (1, 3):
        _compare(gt, pred, search_range, 30)


def test_metric_oracle_equals_reference_predicted_negative_polarity():
    """Predicted polarity -1: the oracle keys such an event by a cell no ground-truth window looks up, while the CUDA
    kernel (load_rec) counts it as polarity 0.  The product never emits -1; this row decides which side follows the
    reference."""
    gt = _events(300, 7, 40000)
    pred = _events(260, 8, 40000, neg_polarity=True)
    _compare(gt, pred, 1, 30)
