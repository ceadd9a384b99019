"""The voxelisation convention of events_to_voxels, on cases whose answers are worked out by hand, and the host-side
argument checks of the wrapper (they run before anything touches a device)."""
import numpy as np
import pytest

from oracle.voxel_oracle import events_to_voxels_oracle, frame_edges

EV = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])


def _ev(rows, dtype=EV):
    a = np.zeros(len(rows), dtype=dtype)
    for i, r in enumerate(rows):
        a[i] = r
    return a


def _cells(grid):
    """Nonzero cells as {(f, plane, c, y, x): count}."""
    return {tuple(int(v) for v in i): int(grid[tuple(i)]) for i in np.argwhere(grid)}


def test_fps30_edges_are_the_cli_offsets():
    assert frame_edges(4, 30).tolist() == [0, 33333, 66666, 100000, 133333]
    assert frame_edges(3, 30, -5 * 10 ** 11).tolist() == [-5 * 10 ** 11 + v for v in (0, 33333, 66666, 100000)]
    from v2ce_toolbox_b200 import v2ce as drv
    from v2ce_toolbox_b200.voxelize import _frame_edges
    for fps in (1, 24, 30, 60, 120, 1000, 29.97):
        want = [drv.frame_offset_us(i, fps) for i in range(301)]
        assert frame_edges(300, fps).tolist() == want
        for t0 in (0, -5 * 10 ** 11, 17 * 10 ** 14):
            assert _frame_edges(300, fps, t0, None, 10).tolist() == [t0 + v for v in want]


@pytest.mark.parametrize('t0', [0, -5 * 10 ** 11, 17 * 10 ** 14])
def test_frame_edges_bin_starts_and_last_microsecond_at_fps30(t0):
    e = frame_edges(3, 30, t0)                        # frames of 33333, 33333 and 33334 us
    rows = [(t0 + 0, 1, 2, 1),                        # frame 0, first us: bin 0
            (t0 + 3332, 1, 2, 1),                     # last us of bin 0
            (t0 + 3333, 1, 2, 1),                     # bin 1 starts at floor(33333 / 10) = 3333
            (t0 + 29999, 0, 0, 0),                    # bin 9 starts at floor(9 * 33333 / 10) = 29999
            (t0 + 33332, 0, 0, 0),                    # the last us of frame 0: bin 9
            (t0 + 33333, 3, 1, -1),                   # exactly on the edge: frame 1, bin 0
            (t0 + 66666 + 9999, 2, 0, 1),             # frame 2 (33334 us): bin 3 starts at floor(3 * 33334 / 10) = 10000
            (t0 + 66666 + 10000, 2, 0, 1),
            (t0 + 99999, 2, 0, 0)]                    # the last us of the 33334-us frame: bin 9
    grid, status = events_to_voxels_oracle(_ev(rows), e, 10, 4, 3)
    assert status.tolist() == [0, 0, 0, 0]
    assert _cells(grid) == {(0, 0, 0, 2, 1): 2, (0, 0, 1, 2, 1): 1, (0, 1, 9, 0, 0): 2, (1, 1, 0, 1, 3): 1,
                            (2, 0, 2, 0, 2): 1, (2, 0, 3, 0, 2): 1, (2, 1, 9, 0, 2): 1}


@pytest.mark.parametrize('nbins,starts', [(1, [0]),
                                          (9, [0, 3703, 7407, 11111, 14814, 18518, 22222, 25925, 29629]),
                                          (10, [0, 3333, 6666, 9999, 13333, 16666, 19999, 23333, 26666, 29999]),
                                          (16, [0, 2083, 4166, 6249, 8333, 10416, 12499, 14583, 16666, 18749, 20833,
                                                22916, 24999, 27083, 29166, 31249])])
def test_every_bin_start_and_the_microsecond_before_it(nbins, starts):
    """Bin c of a 33333-us frame starts at floor(c * 33333 / nbins) (the starts are written out)."""
    e = np.array([0, 33333], dtype=np.int64)
    ts = sorted(set(starts) | {s - 1 for s in starts[1:]} | {33332})
    grid, status = events_to_voxels_oracle(_ev([(t, 0, 0, 1) for t in ts]), e, nbins, 1, 1)
    assert status.tolist() == [0, 0, 0, 0]
    want = np.zeros(nbins, dtype=np.int64)
    for t in ts:
        want[max(c for c, s in enumerate(starts) if s <= t)] += 1
    assert grid[0, 0, :, 0, 0].tolist() == want.tolist()


def test_closed_form_is_the_last_bin_whose_start_is_reached():
    """((r + 1) * nbins - 1) // L is the largest c with floor(c * L / nbins) <= r, also for frames shorter than nbins."""
    rng = np.random.default_rng(3)
    for _ in range(200):
        L = int(rng.choice([1, 2, 5, 7, 33333, 33334, 1_000_000, int(rng.integers(1, 10 ** 6))]))
        nbins = int(rng.integers(1, 20))
        r = np.unique(np.concatenate([rng.integers(0, L, 50), [0, L - 1]]))
        grid, _ = events_to_voxels_oracle(_ev([(int(t), 0, 0, 1) for t in r]), np.array([0, L]), nbins, 1, 1)
        want = np.zeros(nbins, dtype=np.int64)
        for t in r:
            want[max(c for c in range(nbins) if (c * L) // nbins <= t)] += 1
        assert grid[0, 0, :, 0, 0].tolist() == want.tolist(), (L, nbins)


def test_uneven_edges():
    e = np.array([10, 15, 100, 101], dtype=np.int64)  # frames of 5, 85 and 1 us
    rows = [(10, 0, 0, 1),                            # L = 5 < nbins: bins 0 and 1 both start at 10 -> bin 1
            (14, 0, 0, 1),                            # r = 4: bin ((5 * 10) - 1) // 5 = 9
            (15, 0, 0, 1),                            # frame 1, bin 0
            (15 + 42, 0, 0, 1),                       # r = 42: starts floor(c * 85 / 10) = ..., 34, 42, 51 -> bin 5
            (15 + 41, 0, 0, 1),                       # bin 4
            (100, 0, 0, 1)]                           # a 1-us frame: bin 9
    grid, status = events_to_voxels_oracle(_ev(rows), e, 10, 1, 1)
    assert status.tolist() == [0, 0, 0, 0]
    assert _cells(grid) == {(0, 0, 1, 0, 0): 1, (0, 0, 9, 0, 0): 1, (1, 0, 0, 0, 0): 1, (1, 0, 5, 0, 0): 1,
                            (1, 0, 4, 0, 0): 1, (2, 0, 9, 0, 0): 1}


def test_polarity_sensor_and_time_range_status():
    e = frame_edges(2, 30)
    rows = [(5, 1, 1, 1), (5, 1, 1, 0), (5, 1, 1, -1),          # planes 0, 1, 1
            (5, 1, 1, 2), (5, 1, 1, -2),                        # polarity -> status[1]
            (5, 4, 0, 1), (5, -1, 0, 1), (5, 0, 3, 1), (5, 0, -1, 1),   # outside a 4 x 3 sensor -> status[0]
            (5, 9, 9, 7),                                       # outside the sensor is counted first
            (-1, 0, 0, 1), (66666, 0, 0, 0), (10 ** 12, 0, 0, 2)]    # before / at the end / bad polarity wins
    grid, status = events_to_voxels_oracle(_ev(rows), e, 10, 4, 3)
    assert status.tolist() == [5, 3, 1, 1]
    assert _cells(grid) == {(0, 0, 0, 1, 1): 1, (0, 1, 0, 1, 1): 2}


def test_any_integer_widths_and_chunking():
    wide = np.dtype([('timestamp', '<i8'), ('x', '<i4'), ('y', '<u2'), ('polarity', '<i8')])
    rng = np.random.default_rng(0)
    n = 5000
    ev = np.zeros(n, dtype=wide)
    ev['timestamp'] = rng.integers(-100, 70000, n)
    ev['x'] = rng.integers(-2, 12, n)
    ev['y'] = rng.integers(0, 9, n)
    ev['polarity'] = rng.integers(-2, 3, n)
    e = frame_edges(2, 30)
    a, sa = events_to_voxels_oracle(ev, e, 9, 10, 8)
    b, sb = events_to_voxels_oracle(ev.astype(EV), e, 9, 10, 8, chunk=333)
    assert np.array_equal(a, b) and np.array_equal(sa, sb)
    assert int(a.sum()) + int(sa.sum()) == n


def test_wrapper_rejects_bad_arguments_on_the_host():
    from v2ce_toolbox_b200 import V2ceError, events_to_voxels
    ev = _ev([(5, 1, 1, 1)])
    with pytest.raises(V2ceError):
        events_to_voxels(ev, 2, device='cpu')
    with pytest.raises(ValueError, match='exactly one'):
        events_to_voxels(ev)
    with pytest.raises(ValueError, match='exactly one'):
        events_to_voxels(ev, 2, frame_edges_us=[0, 1, 2])
    with pytest.raises(ValueError, match='strictly increasing'):
        events_to_voxels(ev, frame_edges_us=[0, 5, 5])
    with pytest.raises(ValueError, match='strictly increasing'):
        events_to_voxels(ev, frame_edges_us=[0, 5, 3])
    with pytest.raises(ValueError, match='F \\+ 1'):
        events_to_voxels(ev, frame_edges_us=[0])
    with pytest.raises(ValueError, match='int64 bin'):
        events_to_voxels(ev, frame_edges_us=[-(1 << 61), 1 << 61], nbins=2)
    with pytest.raises(ValueError, match='n_frames'):
        events_to_voxels(ev, 0)
    with pytest.raises(ValueError, match='nbins'):
        events_to_voxels(ev, 2, nbins=0)
    with pytest.raises(ValueError, match='fps'):
        events_to_voxels(ev, 2, fps=0)
    wide = np.dtype([('timestamp', '<i8'), ('x', '<i4'), ('y', '<i4'), ('polarity', '<i4')])
    with pytest.raises(IndexError):                   # 65541 would wrap to x = 5 in the packed int16 field
        events_to_voxels(_ev([(5, 65541, 1, 1)], wide), 2)
    with pytest.raises(ValueError, match='polarity'):  # 257 would wrap to 1 in the packed int8 field
        events_to_voxels(_ev([(5, 1, 1, 257)], wide), 2)
