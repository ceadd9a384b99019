"""events_to_voxels -- numpy restatement of the toolbox's voxelisation convention (v2ce_toolbox_b200/voxelize.py,
include/v2ce_b200.h v2ce_events_to_voxels).

TEST INFRASTRUCTURE (see oracle/__init__.py).  This convention is the toolbox's own; it is not the reference's training
voxeliser and is not checked against it.  Per event, in this order: outside the sensor -> status[0]; polarity 1 ->
plane 0, 0 / -1 -> plane 1, anything else -> status[1]; t < e[0] -> status[2]; t >= e[F] -> status[3]; else frame
f = searchsorted(e, t, 'right') - 1, bin c = ((t - e[f] + 1) * nbins - 1) // (e[f+1] - e[f]) in int64, and
voxels[f, plane, c, y, x] += 1 (np.bincount over the flat cell index, chunked so that 10^8 events fit in memory)."""
import numpy as np


def events_to_voxels_oracle(events, frame_edges_us, nbins, width, height, chunk=1 << 24):
    """events: record array (timestamp, x, y, polarity; any integer widths).  Returns (int64 (F, 2, nbins, H, W),
    int64[4] status counts)."""
    edges = np.asarray(frame_edges_us, dtype=np.int64)
    F = edges.shape[0] - 1
    assert F >= 1 and (np.diff(edges) > 0).all()
    cells = F * 2 * nbins * height * width
    grid = np.zeros(cells, dtype=np.int64)
    status = np.zeros(4, dtype=np.int64)
    n = len(events)
    for s in range(0, n, chunk):
        ev = events[s:s + chunk]
        t = np.asarray(ev['timestamp']).astype(np.int64)
        x = np.asarray(ev['x']).astype(np.int64)
        y = np.asarray(ev['y']).astype(np.int64)
        p = np.asarray(ev['polarity']).astype(np.int64)
        inside = (x >= 0) & (x < width) & (y >= 0) & (y < height)
        status[0] += int((~inside).sum())
        pol_ok = (p == 1) | (p == 0) | (p == -1)
        status[1] += int((inside & ~pol_ok).sum())
        ok = inside & pol_ok
        status[2] += int((ok & (t < edges[0])).sum())
        status[3] += int((ok & (t >= edges[-1])).sum())
        ok &= (t >= edges[0]) & (t < edges[-1])
        t, x, y, p = t[ok], x[ok], y[ok], p[ok]
        f = np.searchsorted(edges, t, side='right') - 1
        r = t - edges[f]
        length = edges[f + 1] - edges[f]
        c = ((r + 1) * nbins - 1) // length
        plane = np.where(p == 1, 0, 1)
        idx = (((f * 2 + plane) * nbins + c) * height + y) * width + x
        grid += np.bincount(idx, minlength=cells)
    return grid.reshape(F, 2, nbins, height, width), status


def frame_edges(n_frames, fps, t0_us=0):
    """e[f] = t0_us + int(f / fps * 1e6), f = 0..n_frames, each in Python float arithmetic (v2ce.py:365)."""
    return np.array([t0_us + int(f * 1 / fps * 1e6) for f in range(n_frames + 1)], dtype=np.int64)
