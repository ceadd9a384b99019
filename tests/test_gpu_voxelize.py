"""events_to_voxels on the B200: bit for bit against oracle/voxel_oracle.py on a poisoned output, independent of the
record order, and round trips through the samplers whose output it voxelises (LDATI, 'even' / 'random').

The round trips compare the voxelised grid with the counts the samplers were given.  A sampler places an event in its
bin by float32 arithmetic, the voxeliser by exact integer bin starts, so an event within a few microseconds of a bin
boundary can land in the neighbouring bin.  `_explain_by_boundary_events` accepts a difference only when events that
sit that close to the boundary, in the direction of the move, account for every unit of it."""
import numpy as np
import pytest
import torch

from conftest import record_measurement
from oracle import synth
from oracle.voxel_oracle import events_to_voxels_oracle, frame_edges

pytestmark = pytest.mark.gpu

EV = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])
H, W = 260, 346
PAIRS = 64


def _lib_call(rec_dev, n, edges, nbins, h, w):
    """The C ABI on an output poisoned with 0xFF bytes (NaN) and a poisoned status: returns (grid, status) on the host."""
    from v2ce_toolbox_b200 import _lib
    lib = _lib.load()
    F = len(edges) - 1
    e = torch.from_numpy(np.asarray(edges, dtype=np.int64)).cuda()
    vox = torch.full((F * 2 * nbins * h * w * 4,), 0xFF, dtype=torch.uint8, device='cuda').view(torch.float32)
    status = torch.full((4,), -7, dtype=torch.int64, device='cuda')
    _lib.check(lib.v2ce_events_to_voxels(_lib.ptr(rec_dev) if n else None, n, _lib.ptr(e), F, nbins, h, w, _lib.ptr(vox),
                                         _lib.ptr(status), _lib.stream_ptr()))
    return vox.view(F, 2, nbins, h, w), status.cpu().numpy()


def _assert_matches_oracle(rec_dev, edges, nbins, h, w):
    n = rec_dev.numel() // 13
    got, status = _lib_call(rec_dev, n, edges, nbins, h, w)
    host = rec_dev.cpu().numpy().view(EV)
    want, want_status = events_to_voxels_oracle(host, edges, nbins, w, h)
    assert status.tolist() == want_status.tolist()
    g = got.cpu().numpy()
    assert np.array_equal(g, want.astype(np.float32)), (int(np.isnan(g).sum()), float(np.abs(g - want).max()))
    return got, want, status


def _dev(ev):
    return torch.from_numpy(np.ascontiguousarray(ev).view(np.uint8).reshape(-1)).cuda()


def _gt_like(n, F, fps, t0, w, h, seed, bad=False):
    """A shuffled ground-truth-like stream: a moving blob plus noise, a hot pixel, polarities -1 / 0 / 1, some events
    outside the frame range; with bad=True also events outside the sensor and polarity 2."""
    rng = np.random.default_rng(seed)
    span = int(F / fps * 1e6)
    ev = np.zeros(n, dtype=EV)
    ev['timestamp'] = t0 + rng.integers(-span // 50 - 1, span + span // 50 + 2, n)
    cx = (ev['timestamp'] - t0) / max(span, 1) * w
    ev['x'] = np.clip(np.round(cx + rng.normal(0, max(w / 20, 0.5), n)), 0, w - 1)
    ev['y'] = np.clip(np.round(rng.normal(h / 2, max(h / 6, 0.5), n)), 0, h - 1)
    hot = rng.random(n) < 0.05
    ev['x'][hot], ev['y'][hot] = w // 3, h // 2
    ev['polarity'] = rng.choice(np.array([-1, 0, 1], dtype=np.int8), n)
    if bad:
        k = rng.choice(n, n // 100, replace=False)
        ev['x'][k[::3]] = rng.choice([-1, w, 30000], k[::3].size)
        ev['y'][k[1::3]] = rng.choice([-5, h], k[1::3].size)
        ev['polarity'][k[2::3]] = 2
    return ev


# ---- model streams (stream_clip, device route) ------------------------------------------------------------------------
MODELS = [(0, 'reference'), (31, 'lively'), (7, 'lively')]


def _model(seed, init):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(seed, init))
    return m.eval().cuda()


@pytest.fixture(scope='module')
def model_stream():
    """(seed, init) -> (events on the device, voxels of the same model (PAIRS, 2, 10, H, W) on the host) for a
    65-frame clip; one model per route, since the spectral-norm state advances with every call."""
    from v2ce_toolbox_b200 import v2ce as drv
    cache = {}

    def get(seed, init):
        if (seed, init) not in cache:
            frames = synth.make_video(PAIRS + 1, H, W, seed=0)
            res = drv.stream_clip(_model(seed, init), vidcap=synth.FakeVideoReader(frames), batch_size=4, fps=30,
                                  seed=5, write_event_frames=False, events_to_host=False)
            assert res.n_pairs == PAIRS
            vox = drv.video_to_voxels(_model(seed, init), vidcap=synth.FakeVideoReader(frames), batch_size=4)
            cache[(seed, init)] = (res.event_stream_dev, vox)
        return cache[(seed, init)]
    yield get
    cache.clear()


@pytest.mark.parametrize('nbins', [9, 10])
@pytest.mark.parametrize('seed,init', MODELS)
def test_model_stream_bit_exact(model_stream, seed, init, nbins):
    ev, _ = model_stream(seed, init)
    assert ev.numel() > 0
    _, want, status = _assert_matches_oracle(ev, frame_edges(PAIRS, 30), nbins, H, W)
    assert status[0] == status[1] == status[2] == 0
    record_measurement('voxelize_model_stream', init=init, seed=seed, nbins=nbins, events=ev.numel() // 13,
                       at_or_after_last_edge=int(status[3]), max_cell=int(want.max()))


# ---- shuffled GT-like streams over sensors, frame rates and time bases ---------------------------------------------
@pytest.mark.parametrize('w,h,fps,t0,F,n', [
    (346, 260, 30, 0, 64, 3_000_000),
    (346, 260, 30, -5 * 10 ** 11, 20, 1_000_000),
    (346, 260, 1, 17 * 10 ** 14, 3, 2_000_000),
    (346, 260, 1000, 0, 100, 1_000_000),
    (1920, 1080, 30, 17 * 10 ** 14, 4, 4_000_000),
    (1920, 1080, 1000, -5 * 10 ** 11, 3, 500_000),
    (1, 1, 30, 0, 64, 200_000),
    (1, 1, 1000, 17 * 10 ** 14, 7, 300_000),
    (7, 1, 1, -5 * 10 ** 11, 5, 200_000),
    (7, 1, 30, 0, 1, 100_000),
    (5, 3, 1000, 17 * 10 ** 14, 2500, 1_000_000),         # F >= 2000: twelve steps of the frame search
])
@pytest.mark.parametrize('nbins', [9, 10])
def test_gt_like_streams_bit_exact(w, h, fps, t0, F, n, nbins):
    ev = _gt_like(n, F, fps, t0, w, h, seed=F + n)
    _, _, status = _assert_matches_oracle(_dev(ev), frame_edges(F, fps, t0), nbins, h, w)
    assert status[2] > 0 and status[3] > 0 and status[0] == status[1] == 0


@pytest.mark.parametrize('nbins', [1, 10, 16])
def test_invalid_records_are_counted_not_added(nbins):
    ev = _gt_like(500_000, 30, 30, 0, W, H, seed=4, bad=True)
    _, _, status = _assert_matches_oracle(_dev(ev), frame_edges(30, 30), nbins, H, W)
    assert (status > 0).all()


@pytest.mark.parametrize('t0', [0, -5 * 10 ** 11, 17 * 10 ** 14])
def test_uneven_edges_bit_exact(t0):
    rng = np.random.default_rng(2)
    gaps = rng.choice([1, 3, 9, 10, 11, 33333, 33334, 40000, 10 ** 6], 300)
    edges = t0 + np.concatenate([[0], np.cumsum(gaps)]).astype(np.int64)
    ev = np.zeros(2_000_000, dtype=EV)
    ev['timestamp'] = rng.integers(edges[0] - 100, edges[-1] + 100, ev.size)
    ev['timestamp'][::7] = rng.choice(edges, ev[::7].size) + rng.integers(-1, 2, ev[::7].size)   # on and beside edges
    ev['x'], ev['y'] = rng.integers(0, 40, ev.size), rng.integers(0, 30, ev.size)
    ev['polarity'] = rng.choice(np.array([-1, 0, 1], dtype=np.int8), ev.size)
    for nbins in (9, 10):
        _assert_matches_oracle(_dev(ev), edges, nbins, 30, 40)


def test_no_events_write_zeros():
    got, status = _lib_call(None, 0, frame_edges(3, 30), 10, H, W)
    assert status.tolist() == [0, 0, 0, 0] and int(torch.count_nonzero(got)) == 0
    from v2ce_toolbox_b200 import events_to_voxels
    v = events_to_voxels(np.zeros(0, dtype=EV), 3)
    assert v.shape == (3, 2, 10, H, W) and int(torch.count_nonzero(v)) == 0


def test_unaligned_device_records():
    """Records that do not start on a 16-byte boundary (a slice of a larger buffer) give the same counts."""
    ev = _gt_like(1_000_001, 10, 30, 0, W, H, seed=9)
    buf = _dev(ev)
    sub = buf[13:]
    assert sub.data_ptr() % 16 != 0
    _assert_matches_oracle(sub, frame_edges(10, 30), 10, H, W)


def test_order_independence_and_repeatability():
    ev = _gt_like(4_000_000, 32, 30, 0, W, H, seed=1)
    ev = ev[np.argsort(ev['timestamp'], kind='stable')]          # time-ordered like a recording ...
    perm = np.random.default_rng(0).permutation(ev.size)         # ... and shuffled
    from v2ce_toolbox_b200 import events_to_voxels
    a = events_to_voxels(_dev(ev), 32)
    b = events_to_voxels(_dev(ev), 32)
    c = events_to_voxels(_dev(ev[perm]), 32)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert torch.equal(a.view(torch.int32), c.view(torch.int32))
    want, _ = events_to_voxels_oracle(ev, frame_edges(32, 30), 10, W, H)
    assert np.array_equal(a.cpu().numpy(), want.astype(np.float32))


# ---- round trips through the samplers ---------------------------------------------------------------------------------
def _lookup(keys, counts, q):
    if keys.size == 0:
        return np.zeros(q.shape, np.int64)
    i = np.minimum(np.searchsorted(keys, q), keys.size - 1)
    return np.where(keys[i] == q, counts[i], 0)


def _explain_by_boundary_events(got, want, host_ev, edges, nbins, h, w, windows=(1, 2, 4, 8, 16, 32, 64)):
    """got, want: int64 (F, 2, nbins, H, W).  Walks each (plane, pixel) through its slots (frame, bin) in time order:
    s[j] = events that moved from slot j into slot j + 1 (negative: from j + 1 into j; the slot after the last is
    'at or after the last edge').  A forward move must be matched by that many events in slot j + 1 within `win` us of
    its start, a backward move by events in slot j within `win` us of its end.  Returns the smallest window that
    explains every move, and the moves: forward, backward, and across frame edges (forward only)."""
    F = len(edges) - 1
    S = F * nbins
    d = (got - want).transpose(1, 3, 4, 0, 2).reshape(2 * h * w, S)
    s = -np.cumsum(d, axis=1)
    rows, cols = np.nonzero(s)
    moves = s[rows, cols]
    if rows.size == 0:
        return 0, 0, 0, 0
    t = host_ev['timestamp'].astype(np.int64)
    x, y, p = host_ev['x'].astype(np.int64), host_ev['y'].astype(np.int64), host_ev['polarity'].astype(np.int64)
    e = np.asarray(edges, dtype=np.int64)
    ok = (x >= 0) & (x < w) & (y >= 0) & (y < h) & (p >= -1) & (p <= 1) & (t >= e[0])
    t, x, y, p = t[ok], x[ok], y[ok], p[ok]
    row = (np.where(p == 1, 0, 1) * h + y) * w + x
    f = np.minimum(np.searchsorted(e, t, side='right') - 1, F)
    inside = f < F
    fi = np.minimum(f, F - 1)
    L = e[fi + 1] - e[fi]
    c = np.where(inside, ((t - e[fi] + 1) * nbins - 1) // L, 0)
    slot = np.where(inside, fi * nbins + c, S)
    start = np.where(inside, e[fi] + (c * L) // nbins, e[F])
    end = np.where(inside, e[fi] + ((c + 1) * L) // nbins, np.iinfo(np.int64).max)
    for win in windows:
        fwd = (t - start < win) & (slot >= 1)          # may have come from the slot before
        bwd = (end - t <= win) & (slot < S - 1)        # may belong to the slot after
        kf, nf = np.unique(row[fwd] * (S + 1) + slot[fwd] - 1, return_counts=True)
        kb, nb = np.unique(row[bwd] * (S + 1) + slot[bwd], return_counts=True)
        key = rows.astype(np.int64) * (S + 1) + cols
        if ((moves > 0) & (moves > _lookup(kf, nf, key))).any() or ((moves < 0) & (-moves > _lookup(kb, nb, key))).any():
            continue
        at_edge = (cols + 1) % nbins == 0
        assert (moves[at_edge] >= 0).all(), 'an event moved back across a frame edge'
        return win, int(moves[moves > 0].sum()), int(-moves[moves < 0].sum()), int(moves[at_edge].sum())
    raise AssertionError(f'{int(np.abs(moves).sum())} moved events are not explained by events within '
                         f'{windows[-1]} us of a bin boundary')


@pytest.mark.parametrize('seed,init', MODELS)
def test_round_trip_through_ldati(model_stream, seed, init):
    """LDATI emits max(n, 0) events in bin c of the 9 relocated bins (v2ce_ldati_relocate / relocate_counts): the
    voxelised stream must give those counts back, up to events at a bin boundary."""
    from oracle.ldati_oracle import relocate_counts
    from v2ce_toolbox_b200 import events_to_voxels
    ev, vox = model_stream(seed, init)
    got = events_to_voxels(ev, PAIRS, 30, nbins=9).cpu().numpy().astype(np.int64)
    n, _ = relocate_counts(vox)
    want = np.maximum(n, 0)
    host = ev.cpu().numpy().view(EV)
    assert int(want.sum()) == host.size
    # per (frame, plane, pixel): equal, except events that reached the next frame's start
    per_frame = got.sum(axis=2) - want.sum(axis=2)
    win, fwd, bwd, across = _explain_by_boundary_events(got, want, host, frame_edges(PAIRS, 30), 9, H, W)
    assert win <= 64
    beyond = int((host['timestamp'] >= frame_edges(PAIRS, 30)[-1]).sum())
    assert int(np.abs(per_frame).sum()) <= 2 * across + beyond
    record_measurement('voxelize_ldati_round_trip', init=init, seed=seed, fps=30, events=int(host.size),
                       window_us=win, moved_forward=fwd, moved_backward=bwd, across_frame_edges=across,
                       at_or_after_last_edge=beyond, differing_cells=int(np.count_nonzero(got - want)))


@pytest.mark.parametrize('mode', ['even', 'random'])
@pytest.mark.parametrize('fps', [30, 1000])
def test_round_trip_through_baseline_samplers(mode, fps):
    from v2ce_toolbox_b200 import events_to_voxels
    from v2ce_toolbox_b200.ldati import frame_offsets_us
    from v2ce_toolbox_b200.sample_methods.random_even_sample import sample_voxel_baseline
    F = 16
    kind = 'randint' if mode == 'even' else 'mixed'
    v = synth.make_voxels(kind, F, H, W, seed=fps)
    lists = sample_voxel_baseline(torch.from_numpy(v).cuda(), fps=fps, even=mode == 'even', random=mode == 'random',
                                  seed=3)
    off = frame_offsets_us(0, F, fps)
    edges = frame_edges(F + 1, fps)                   # one frame more: the last frame's late events stay in the grid
    ev = np.concatenate(lists).copy()
    ev['timestamp'] += np.repeat(off, [len(a) for a in lists])
    g = events_to_voxels(_dev(ev), F + 1, fps, nbins=10).cpu().numpy().astype(np.int64)
    # no event is dropped; frame f receives the events of list f except those at or after the next frame's start
    late = [int((a['timestamp'].astype(np.int64) + o >= edges[f + 1]).sum()) for f, (a, o) in enumerate(zip(lists, off))]
    assert int(g.sum()) == ev.size
    for f in range(F + 1):
        assert int(g[f].sum()) == (len(lists[f]) - late[f] if f < F else 0) + (late[f - 1] if f else 0), f
    record_measurement('voxelize_baseline_round_trip', mode=mode, fps=fps, events=int(ev.size),
                       at_or_after_next_frame=int(sum(late)))
    if mode == 'even':
        want = np.concatenate([v, np.zeros_like(v[:1])]).astype(np.int64)
        win, fwd, bwd, across = _explain_by_boundary_events(g, want, ev, edges, 10, H, W)
        assert win <= 64 and across == sum(late)
        record_measurement('voxelize_even_round_trip', fps=fps, window_us=win, moved_forward=fwd, moved_backward=bwd)


# ---- wrapper routes ---------------------------------------------------------------------------------------------------
def test_wrapper_routes_and_errors():
    from v2ce_toolbox_b200 import V2ceError, events_to_voxels
    ev = _gt_like(200_000, 8, 30, 0, W, H, seed=5)
    want, _ = events_to_voxels_oracle(ev, frame_edges(8, 30), 10, W, H)
    want = want.astype(np.float32)
    wide = np.dtype([('timestamp', '<i8'), ('x', '<i4'), ('y', '<u2'), ('polarity', '<i8')])
    for arr in (ev, ev.astype(wide), ev.view(np.recarray)):
        assert np.array_equal(events_to_voxels(arr, 8).cpu().numpy(), want)
    assert np.array_equal(events_to_voxels(_dev(ev), 8).cpu().numpy(), want)
    assert np.array_equal(events_to_voxels(_dev(ev), frame_edges_us=frame_edges(8, 30)).cpu().numpy(), want)
    assert np.array_equal(events_to_voxels(_dev(ev).view(-1, 13), 8).cpu().numpy(), want)   # any uint8 shape
    t0 = 17 * 10 ** 14
    shifted = ev.copy()
    shifted['timestamp'] += t0
    assert np.array_equal(events_to_voxels(shifted, 8, t0_us=t0).cpu().numpy(), want)
    out = ev.copy()
    out['x'][3] = W
    with pytest.raises(IndexError):
        events_to_voxels(out, 8)
    bad = ev.copy()
    bad['polarity'][5] = 2
    with pytest.raises(ValueError):
        events_to_voxels(_dev(bad), 8)
    with pytest.raises(ValueError):
        events_to_voxels(ev, frame_edges_us=[0, 10, 10, 20])
    with pytest.raises(V2ceError):
        events_to_voxels(_dev(ev).cpu(), 8)
    with pytest.raises(V2ceError):
        events_to_voxels(_dev(ev)[:-1], 8)                  # not a whole number of records
