"""oracle.metric_oracle.ts_diff_exact (the vectorised reference the GPU metric is compared with at millions of events,
tests/test_gpu_metric_scale.py) against the per-event ts_diff_metric_oracle, which tests/test_metric_oracle_live.py pins
to the reference function.  CPU only.

The mutation test shows that the planted inputs the GPU rows use tell a correct answer from five plausible kernel
errors, each made by a switch of nearest_distances / totals."""
import numpy as np
import pytest

from oracle import metric_oracle as mo

SENSORS = [(346, 260), (260, 346), (1920, 1080), (33, 47), (1, 1), (1, 7), (7, 1)]
FPS = [30, 100, 1, 0.3, 0.25, 0.1]
T_BASES = [0, -5 * 10 ** 11, 1_700_000_000_000_000]        # zero, negative, epoch microseconds


def _agree(gt, pred, r, fps, width=346, height=260):
    total, over = mo.ts_diff_exact(gt, pred, r, fps, width, height)
    want = mo.ts_diff_metric_oracle(gt, pred, search_range=r, fps=fps, width=width, height=height)
    cap = 1e6 / fps / 10 * 3
    assert over == want[1]
    assert abs((total + over * cap) / len(gt) - want[0]) <= 1e-12 * max(abs(want[0]), 1.0)
    return total, over


def _random(n, seed, width, height, spread, box=None, neg_polarity=False):
    rng = np.random.default_rng(seed)
    (x0, x1), (y0, y1) = box or ((0, width), (0, height))
    p = rng.integers(0, 2, n)
    if neg_polarity:
        p[p == 0] = -1
    return mo._records(rng.integers(0, spread, n), rng.integers(x0, x1, n), rng.integers(y0, y1, n), p)


def test_caps_of_the_time_matrix():
    """The caps the planted distances sit on: exact at 30 / 100 / 1 fps, at or above 1e6 from 0.3 fps down."""
    assert 1e6 / 30 / 10 * 3 == 10000.0 and 1e6 / 100 / 10 * 3 == 3000.0 and 1e6 / 1 / 10 * 3 == 300000.0
    assert 1e6 / 0.3 / 10 * 3 > 1e6 and 1e6 / 0.25 / 10 * 3 == 1.2e6 and 1e6 / 0.1 / 10 * 3 >= 3e6 - 1e-6


@pytest.mark.parametrize('width,height', SENSORS)
@pytest.mark.parametrize('r', [0, 1, 2, 5])
def test_exact_equals_oracle_planted_edges(width, height, r):
    gt, pred = mo.planted_edges(width, height, r, seed=r, n_background=200)
    for fps in (30, 0.25):
        _agree(gt, pred, r, fps, width, height)


@pytest.mark.parametrize('width,height', [(33, 47), (1, 7), (7, 1), (1, 1)])
def test_exact_equals_oracle_range_63(width, height):
    gt, pred = mo.planted_edges(width, height, 63, seed=5, n_background=100)
    _agree(gt, pred, 63, 30, width, height)


@pytest.mark.parametrize('fps', FPS)
@pytest.mark.parametrize('t_base', T_BASES)
def test_exact_equals_oracle_planted_times(fps, t_base):
    gt, pred = mo.planted_times(fps, 1, seed=7, t_base=t_base, n_empty=6)
    total, over = _agree(gt, pred, 1, fps)
    d = mo.nearest_distances(gt, pred, 1)
    assert (d == mo.NONE).sum() == 6                              # the empty windows are empty
    assert set(mo.planted_distances(fps)) <= set(d[d != mo.NONE].tolist())
    _agree(gt, pred, 0, fps)


@pytest.mark.parametrize('r,fps', [(0, 30), (1, 0.25), (2, 30), (3, 1), (2, 0.3)])
def test_exact_equals_oracle_random(r, fps):
    """Dense random events in a box, with gt polarity -1 and gt times beyond the predicted ones on both sides; and events
    over the whole sensor at a wide time spread (empty and far windows)."""
    gt = _random(4000, 1, 346, 260, 60000, box=((90, 130), (40, 80)), neg_polarity=True)
    gt['timestamp'] -= 20000                                    # some before, some after every predicted event
    gt['timestamp'][::2] += 40000
    pred = _random(3000, 2, 346, 260, 60000, box=((88, 132), (38, 82)))
    _agree(gt, pred, r, fps)
    gt = _random(3000, 3, 346, 260, 5 * 10 ** 7)
    pred = _random(30000, 4, 346, 260, 5 * 10 ** 7)
    _agree(gt, pred, r, fps)


def test_exact_ignores_what_no_window_reaches():
    """Predicted events outside the sensor or with polarity -1 / 2 are never found (the per-event oracle keys them by
    cells no ground-truth window looks up); ground-truth events outside the sensor see the clamped window."""
    gt, pred = mo.planted_edges(33, 47, 2, seed=9, n_background=300)
    extra = mo._records([5, 6, 7, 8, 9], [-1, 33, 3, 4, 5], [4, 5, 47, 6, 7], [0, 1, 0, -1, 2])
    far = mo._records([0, 1, 2], [-2, 35, 3], [3, 4, 48], [0, 1, 0])
    base = _agree(gt, pred, 2, 30, 33, 47)
    assert _agree(gt, np.concatenate([pred, extra]), 2, 30, 33, 47) == base
    _agree(np.concatenate([gt, far]), pred, 2, 30, 33, 47)


def test_exact_scale_smoke():
    """5 000 ground-truth events against 200 000 predicted ones at r = 2 agree with the per-event oracle."""
    gt = _random(5000, 11, 346, 260, 2 * 10 ** 6, neg_polarity=True)
    pred = _random(200000, 12, 346, 260, 2 * 10 ** 6)
    _agree(gt, pred, 2, 30)


def _planted_cases():
    for width, height in SENSORS:
        for r in (0, 1, 2, 5):
            yield ('edges', width, height, r), mo.planted_edges(width, height, r, seed=r), 30
    for fps in FPS:
        yield ('times', fps), mo.planted_times(fps, 1, seed=7, n_empty=6), fps


MUTATIONS = {
    'window one pixel short on the high side': (dict(window_hi=0), {}),
    'width and height swapped in the clamps': (dict(swap_clamps=True), {}),
    'a tie at the cap counted as overflow': ({}, dict(tie_overflows=True)),
    'the 1e6 clamp dropped': ({}, dict(clamp=False)),
    'polarity ignored': (dict(polarity=False), {}),
}


@pytest.mark.parametrize('name', list(MUTATIONS))
def test_mutations_are_rejected(name):
    """Every variant disagrees with the correct reference on each planted row it must be visible on: the window and
    polarity errors on every edge row with a neighbour to miss, the swap on every W != H row, the tie at 30 / 100 / 1
    fps, the clamp at 0.3 / 0.25 / 0.1 fps."""
    near_kw, tot_kw = MUTATIONS[name]
    missed = []
    for key, (gt, pred), fps in _planted_cases():
        r = key[3] if key[0] == 'edges' else 1
        w, h = key[1:3] if key[0] == 'edges' else (346, 260)
        want = mo.ts_diff_exact(gt, pred, r, fps, w, h)
        got = mo.totals(mo.nearest_distances(gt, pred, r, w, h, **near_kw), fps, **tot_kw)
        if got == want:
            missed.append(key)
    if name.startswith('window'):
        must = [k for k, _, _ in _planted_cases() if k[0] == 'edges' and (k[1] > 1 or k[2] > 1 or k[3] == 0)]
    elif name.startswith('width'):
        must = [k for k, _, _ in _planted_cases() if k[0] == 'edges' and k[1] != k[2]]
    elif name.startswith('a tie'):
        must = [('times', f) for f in (30, 100, 1)]
    elif name.startswith('the 1e6'):
        must = [('times', f) for f in (0.3, 0.25, 0.1)]
    else:
        must = [k for k, _, _ in _planted_cases() if k[0] == 'edges']
    assert must and not set(must) & set(missed), f'{name}: not rejected on {sorted(set(must) & set(missed), key=str)}'
