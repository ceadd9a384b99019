"""ts_diff_metric (csrc/metrics.cu) at recording scale and at its edges, exactly.

v2ce_ts_diff_metric returns an exact int64 total and an exact overflow count, so every row here calls it through the C
ABI and compares result[0..3] as integers with oracle.metric_oracle.ts_diff_exact, which tests/test_metric_exact_reference.py
checks against the per-event oracle (and tests/test_metric_oracle_live.py pins that to the reference).  The planted
inputs give every ground-truth event its own distance, so the total shows which predicted events a window reached and
how a distance next to the cap or the 1e6 clamp was counted; the CPU file shows that a window one pixel short, swapped
width / height clamps, a tie counted as overflow, a dropped 1e6 clamp or ignored polarity each change the answer.

Rows: three model streams of one 64-pair 260x346 clip (1.3-1.8e8 events each), dense cells, the sensor geometry matrix
(346x260, 260x346, 1920x1080, 33x47, 1x1, 1x7, 7x1 at search_range 0, 1, 2, 5 and 63), the time matrix (fps 30,
100, 1, 0.3, 0.25, 0.1 on zero, negative and epoch timestamps), the three input routes of the Python wrapper, and the
limits and errors of the C ABI and the wrapper."""
import ctypes
import time

import numpy as np
import pytest
import torch

from oracle import metric_oracle as mo, synth

pytestmark = pytest.mark.gpu

EVENT_DTYPE = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])
T_BASES = [0, -5 * 10 ** 11, 1_700_000_000_000_000]


def _cap(fps):
    return 1e6 / fps / 10 * 3                    # stage2_metrics.py:73, as the wrapper computes it


def _dev(ev):
    return torch.from_numpy(np.ascontiguousarray(ev).view(np.uint8).reshape(-1).copy()).cuda()


def _metric(gt_dev, pred_dev, r, fps, width=346, height=260):
    """result[0..3] of v2ce_ts_diff_metric as Python ints, on packed uint8 device records."""
    from v2ce_toolbox_b200 import _lib
    from v2ce_toolbox_b200._lib import check, ptr, stream_ptr
    lib = _lib.load()
    n_gt, n_pred = gt_dev.numel() // 13, pred_dev.numel() // 13
    n = ctypes.c_size_t()
    check(lib.v2ce_ts_diff_workspace_bytes(width, height, n_pred, ctypes.byref(n)))
    ws = torch.full((n.value,), 0xFF, dtype=torch.uint8, device='cuda')          # no reliance on a zeroed workspace
    res = torch.full((4,), -7, dtype=torch.int64, device='cuda')
    check(lib.v2ce_ts_diff_metric(ptr(gt_dev), n_gt, ptr(pred_dev), n_pred, width, height, r, _cap(fps), ptr(ws),
                                  ws.numel(), ptr(res), stream_ptr()))
    return [int(v) for v in res.cpu().tolist()]


def _check(gt, pred, r, fps, width=346, height=260):
    """The kernel's integers equal the exact reference's; the wrapper's mean is (total + overflow * cap) / n_gt."""
    from v2ce_toolbox_b200.stage2_metrics import ts_diff_metric
    got = _metric(_dev(gt), _dev(pred), r, fps, width, height)
    total, over = mo.ts_diff_exact(gt, pred, r, fps, width, height)
    assert got == [total, over, 0, 0], (got, total, over)
    mean = ts_diff_metric(gt, pred, search_range=r, fps=fps, width=width, height=height)
    assert mean[1] == over and mean[0] == (total + over * _cap(fps)) / len(gt)
    return total, over


# ---------------------------------------------------------------------------------------------------------------------
# the product: device records of stream_clip
# ---------------------------------------------------------------------------------------------------------------------
def _stream(model, frames, seed, fps):
    from v2ce_toolbox_b200 import v2ce as drv
    res = drv.stream_clip(model, vidcap=synth.FakeVideoReader(frames), seq_len=16, width=346, height=260, fps=fps,
                          seed=seed, write_event_frames=False, events_to_host=False)
    assert res.n_pairs == 64
    return res.event_stream_dev


def _model(seed):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(seed, 'lively'))
    return m.eval().to('cuda')


@pytest.fixture(scope='module')
def streams():
    """Three streams of one 65-frame 260x346 clip.  'gt': model seed 31, LDATI seed 2, 30 fps.  'pred': the same model
    with LDATI seed 1 at 29 fps, so it lies close in time and drifts by 1 149 us a frame (two seeds of one model at
    one frame rate give the same timestamp wherever both place an event).  'other': model seed 32, so distances are
    larger and more events overflow.  Device records, host views and the sorted index of each predicted set."""
    frames = synth.make_video(65, 260, 346, seed=21)
    model = _model(31)
    dev = {'gt': _stream(model, frames, 2, 30), 'pred': _stream(model, frames, 1, 29),
           'other': _stream(_model(32), frames, 1, 30)}
    host = {k: v.cpu().numpy().view(EVENT_DTYPE) for k, v in dev.items()}
    print(f'\nproduct row: {len(host["gt"])} gt, {len(host["pred"])} pred, {len(host["other"])} other-model events')
    assert min(len(v) for v in host.values()) > 10 ** 6
    t0 = time.perf_counter()
    cells = {k: mo.PredCells(host[k]) for k in ('pred', 'other')}
    print(f'  predicted-event index {time.perf_counter() - t0:.1f} s')
    return dev, host, cells


def _gt_subsample(dev, host, step):
    return host['gt'][::step], dev['gt'].view(-1, 13)[::step].contiguous().view(-1)


# The kernel always runs on all predicted events (count, single-block scan and fill over 1.3-1.8e8 of them).  The
# exact reference costs about 0.08 us per (ground-truth event, window offset) plus the sorts, so the ground truth is
# subsampled on the device: every 16th event at r = 0 and 1, every 64th at 2 and every 256th at 5.
PRODUCT_ROWS = [(0, 16), (1, 16), (2, 64), (5, 256)]


@pytest.mark.parametrize('p_name', ['pred', 'other'])
def test_product_clip_streams(streams, p_name):
    dev, host, cells = streams
    for r, step in PRODUCT_ROWS:
        g_host, g_dev = _gt_subsample(dev, host, step)
        t0 = time.perf_counter()
        best = cells[p_name].nearest(g_host, r)
        t_ref = time.perf_counter() - t0
        for fps in (30, 1):
            got = _metric(g_dev, dev[p_name], r, fps)
            want = mo.totals(best, fps)
            assert got == [*want, 0, 0], (p_name, r, fps, got, want)
        print(f'  gt vs {p_name} r={r} 1/{step}: {len(g_host)} gt, fps 1 total {want[0]} overflow {want[1]}, '
              f'{(best == mo.NONE).sum()} empty windows, reference {t_ref:.1f} s')
        total, over = mo.totals(best, 30)
        assert 0 < over < len(g_host) and total > 0                  # at 30 fps both sums are in play


def test_product_clip_streams_fps_0_25(streams):
    """gt against the first quarter (about 16 frames) of the other model's stream at fps 0.25 (cap 1.2e6): a
    ground-truth event of a later frame can have its nearest predicted event more than 1e6 us away, and then adds
    exactly 1e6."""
    dev, host, _ = streams
    g_host, g_dev = _gt_subsample(dev, host, 16)
    n = len(host['other']) // 4                               # records are in frame order: about 16 frames
    best = mo.PredCells(host['other'][:n]).nearest(g_host, 0)
    print(f'\n  gt vs the first {n} other-model events: {(best == mo.NONE).sum()} empty windows, '
          f'{(best > 10 ** 6).sum()} nearest beyond 1e6')
    assert ((best > 10 ** 6) & (best != mo.NONE)).sum() > 0     # empty windows: test_time_matrix (none occur here)
    assert _metric(g_dev, dev['other'][:n * 13], 0, 0.25) == [*mo.totals(best, 0.25), 0, 0]


# ---------------------------------------------------------------------------------------------------------------------
# dense cells, geometry, time
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('r', [0, 1, 2])
def test_dense_cells(r):
    """Thousands of predicted timestamps in each of a few cells (one thread walks all of them, per window cell), ground
    truth in and around them, and empty regions elsewhere."""
    rng = np.random.default_rng(40 + r)
    hot = [(0, 0), (173, 130), (345, 259), (100, 7)]
    t, x, y, p = [], [], [], []
    for hx, hy in hot:
        n = 6000
        t.append(rng.integers(0, 2 * 10 ** 6, n)), x.append(np.full(n, hx)), y.append(np.full(n, hy))
        p.append(rng.integers(0, 2, n))
    pred = mo._records(*(np.concatenate(v) for v in (t, x, y, p)))
    n = 20000
    c = rng.integers(0, len(hot), n)
    hx, hy = np.array(hot)[c].T
    gx = np.clip(hx + rng.integers(-3, 4, n), 0, 345)
    gy = np.clip(hy + rng.integers(-3, 4, n), 0, 259)
    gp = rng.choice([-1, 0, 1], n)                                              # ground-truth -1 counts as 0
    gt = mo._records(rng.integers(-1000, 2 * 10 ** 6 + 1000, n), gx, gy, gp)
    gt = np.concatenate([gt, mo.planted_edges(346, 260, r, seed=r)[0]])        # far from the hot cells: empty windows
    total, over = _check(gt, pred, r, 30)
    assert over > 0 and total > 0


GEOMETRY = [(w, h, r) for w, h in [(346, 260), (260, 346), (1920, 1080), (33, 47), (1, 1), (1, 7), (7, 1)]
            for r in (0, 1, 2, 5)] + [(33, 47, 63), (1, 7, 63), (7, 1, 63), (1, 1, 63), (346, 260, 63)]


@pytest.mark.parametrize('width,height,r', GEOMETRY)
def test_geometry(width, height, r):
    """Every corner and edge middle has ground-truth events with predicted events at offset exactly r and r + 1, each
    at its own distance, plus random events over the sensor.  346x260 has events at x >= 260 (= height), 260x346 at
    y >= 260 (= width): an x / y swap in the clamps shows only there; 1920x1080 has 4.1 M cells for the single-block
    scan (about 4 000 iterations of its loop)."""
    gt, pred = mo.planted_edges(width, height, r, seed=r + width, n_background=20000 if r < 63 else 300)
    if width > height:
        assert (gt['x'] >= height).any() and (pred['x'] >= height).any()
    if height > width:
        assert (gt['y'] >= width).any() and (pred['y'] >= width).any()
    _check(gt, pred, r, 30, width, height)


@pytest.mark.parametrize('fps', [30, 100, 1, 0.3, 0.25, 0.1])
@pytest.mark.parametrize('t_base', T_BASES, ids=['t0', 'negative', 'epoch'])
def test_time_matrix(fps, t_base):
    """Distances 0 and cap - 1, cap, cap + 1 (30, 100, 1 fps: caps 10 000, 3 000, 300 000 exactly), and 999 999, 1e6,
    1e6 + 1, 2e6 plus empty windows where the cap is >= 1e6 (0.3, 0.25, 0.1 fps: each such event adds exactly 1e6)."""
    gt, pred = mo.planted_times(fps, 1, seed=8, t_base=t_base, n_empty=6)
    for r in (0, 1):
        total, over = _check(gt, pred, r, fps)
        if fps <= 0.3:
            assert over == 0 and total == int(mo.nearest_distances(gt, pred, r).clip(max=10 ** 6).sum())


# ---------------------------------------------------------------------------------------------------------------------
# routes, limits, errors
# ---------------------------------------------------------------------------------------------------------------------
def test_routes_give_identical_integers():
    """Packed numpy records, numpy records of other field dtypes (int64 x / y, int32 polarity, -1 for ground truth)
    converted by the wrapper, and uint8 device tensors all give the same integers."""
    from v2ce_toolbox_b200.stage2_metrics import _records_dev, ts_diff_metric
    gt, pred = mo.planted_edges(346, 260, 2, seed=12, n_background=30000)
    wide = np.dtype([('timestamp', '<i8'), ('x', '<i8'), ('y', '<i8'), ('polarity', '<i4')])
    gt_w, pred_w = gt.astype(wide), pred.astype(wide)
    gt_w['polarity'][gt_w['polarity'] == 0] = -1
    want = [*mo.ts_diff_exact(gt, pred, 2, 30), 0, 0]
    outs = []
    for g, p in ((gt, pred), (gt_w, pred_w), (_dev(gt), _dev(pred))):
        g_dev, n_g = _records_dev(g, torch.device('cuda'))
        p_dev, n_p = _records_dev(p, torch.device('cuda'))
        assert (n_g, n_p) == (len(gt), len(pred))
        outs.append(_metric(g_dev, p_dev, 2, 30))
        mean = ts_diff_metric(g, p, search_range=2, fps=30)
        assert mean[1] == want[1] and mean[0] == (want[0] + want[1] * _cap(30)) / len(gt)
    assert outs == [want] * 3


def test_workspace_query_limits():
    """n_pred up to 2^31 - 1 and width * height * 2 below 2^30 (32-bit cell starts and indices inside); queried only."""
    from v2ce_toolbox_b200 import _lib
    lib = _lib.load()
    n = ctypes.c_size_t()
    assert lib.v2ce_ts_diff_workspace_bytes(346, 260, (1 << 31) - 1, ctypes.byref(n)) == 0
    assert n.value >= 8 * ((1 << 31) - 1) + 4 * 3 * 346 * 260 * 2
    assert lib.v2ce_ts_diff_workspace_bytes(346, 260, 1 << 31, ctypes.byref(n)) != 0
    assert lib.v2ce_ts_diff_workspace_bytes(1 << 14, 1 << 15, 1, ctypes.byref(n)) != 0          # 2 * W * H == 2^30
    assert lib.v2ce_ts_diff_workspace_bytes(1 << 14, (1 << 15) - 1, 1, ctypes.byref(n)) == 0
    assert n.value >= 12 * (1 << 14) * ((1 << 15) - 1) * 2
    assert lib.v2ce_ts_diff_workspace_bytes(346, 260, -1, ctypes.byref(n)) != 0
    assert lib.v2ce_ts_diff_workspace_bytes(0, 260, 1, ctypes.byref(n)) != 0


def test_errors():
    """search_range 64 is refused (the reference has no limit; the kernel's windows stop at 63), no ground truth
    divides by zero like the reference, and events outside the sensor raise IndexError."""
    from v2ce_toolbox_b200._lib import V2ceError
    from v2ce_toolbox_b200.stage2_metrics import ts_diff_metric
    gt, pred = mo.planted_edges(33, 47, 2, seed=3)
    with pytest.raises(V2ceError):
        ts_diff_metric(gt, pred, search_range=64, width=33, height=47)
    with pytest.raises(ZeroDivisionError):
        ts_diff_metric(gt[:0], pred, width=33, height=47)
    for field, value in (('x', -1), ('y', 47), ('polarity', 2)):
        for which in ('gt', 'pred'):
            g, p = gt.copy(), pred.copy()
            (g if which == 'gt' else p)[field][3] = value
            with pytest.raises(IndexError):
                ts_diff_metric(g, p, search_range=2, width=33, height=47)
