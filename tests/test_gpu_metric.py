"""GPU ts_diff_metric (csrc/metrics.cu; SURVEY.md 8f N4) against the oracle, which tests/test_metric_oracle_live.py pins
to the reference function (train/scripts/stage2/stage2_metrics.py:22-88).  The overflow count and the integer sum are
exact; the float64 mean is compared to 1e-12 relative (the reference adds the terms one by one in Python floats)."""
import numpy as np
import pytest
import torch

from oracle import metric_oracle as mo

pytestmark = pytest.mark.gpu

EVENT_DTYPE = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])


def _events(n, seed, spread, box=((90, 130), (40, 80)), neg_polarity=False):
    rng = np.random.default_rng(seed)
    ev = np.zeros(n, dtype=EVENT_DTYPE)
    ev['timestamp'] = rng.integers(0, spread, n)
    ev['x'] = rng.integers(*box[0], n)
    ev['y'] = rng.integers(*box[1], n)
    ev['polarity'] = rng.integers(0, 2, n)
    if neg_polarity:
        ev['polarity'][ev['polarity'] == 0] = -1
    return ev


# fps 0.25 / 0.3: the cap is >= 1e6, so the 1 126 (r = 0) and 14 (r = 1) ground-truth events with an empty window add 1e6
@pytest.mark.parametrize('search_range,fps,n', [(0, 30, 2000), (1, 30, 2000), (3, 120, 1500), (0, 30, 1), (0, 0.25, 2000),
                                                (1, 0.3, 2000)])
def test_metric_equals_oracle(search_range, fps, n):
    from v2ce_toolbox_b200.stage2_metrics import ts_diff_metric
    gt = _events(n, 1, 60000, neg_polarity=True)
    pred = _events(max(n - 100, 1), 2, 60000)
    want = mo.ts_diff_metric_oracle(gt, pred, search_range=search_range, fps=fps)
    got = ts_diff_metric(gt, pred, search_range=search_range, fps=fps)
    assert got[1] == want[1]
    assert abs(got[0] - want[0]) <= 1e-12 * max(abs(want[0]), 1.0)
    # the same from packed records already on the device (what the pipeline leaves there)
    dev = torch.from_numpy(pred.view(np.uint8).reshape(-1).copy()).cuda()
    gt0 = gt.copy()
    gt0['polarity'][gt0['polarity'] == -1] = 0
    got2 = ts_diff_metric(torch.from_numpy(gt0.view(np.uint8).reshape(-1).copy()).cuda(), dev, search_range=search_range, fps=fps)
    assert np.array_equal(got, got2)


def test_metric_edges():
    from v2ce_toolbox_b200.stage2_metrics import ts_diff_metric
    gt = _events(50, 3, 1000, box=((0, 3), (257, 260)))                 # sensor corners: the window is clamped
    pred = _events(0, 4, 1000)
    out = ts_diff_metric(gt, pred, search_range=2, fps=30)             # no predicted events: every distance is capped
    assert out[1] == 50 and abs(out[0] - 1e6 / 30 / 10 * 3) < 1e-9
    same = ts_diff_metric(gt, gt, search_range=0, fps=30)
    assert same[0] == 0 and same[1] == 0
    bad = gt.copy()
    bad['x'][0] = 400
    with pytest.raises(IndexError):
        ts_diff_metric(bad, gt)
