"""ts_diff_metric -- CPU restatement of /root/reference/train/scripts/stage2/stage2_metrics.py:22-88.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Vectorised per cell instead of per event, same arithmetic: the smallest
|t_pred - t_gt| over the predicted events of the same polarity within the (clamped) search window, 1e6 when there is
none, capped at 1e6/fps/10*3 with an overflow count; the mean over the ground-truth events.

``ts_diff_metric_oracle`` follows the reference event by event (tests/test_metric_oracle_live.py pins it to the
reference); ``ts_diff_exact`` computes the same thing for millions of events and returns the two integers the CUDA
kernel writes (``nearest_distances`` and ``totals`` are its two halves); ``planted_edges`` / ``planted_times`` build
inputs whose answer shows which predicted events a window reached and how a distance near the cap was counted."""
import numpy as np

NONE = np.iinfo(np.int64).max            # no predicted event in the window
SEP = 10 ** 7                            # time between planted groups: > 1e6 + any planted distance, so groups never mix


def ts_diff_metric_oracle(event_gt, event_pred, search_range=0, fps=30, width=346, height=260):
    gt_p = np.asarray(event_gt['polarity']).astype(np.int64).copy()
    gt_p[gt_p == -1] = 0
    cells = {}
    for t, x, y, p in zip(event_pred['timestamp'], event_pred['x'], event_pred['y'], event_pred['polarity']):
        cells.setdefault((int(x), int(y), int(p)), []).append(int(t))
    cells = {k: np.array(v, dtype=np.int64) for k, v in cells.items()}
    cap = 1e6 / fps / 10 * 3
    total, overflow = 0, 0
    for t, x, y, p in zip(event_gt['timestamp'], event_gt['x'], event_gt['y'], gt_p):
        diff = 1e6
        for a in range(max(int(x) - search_range, 0), min(int(x) + search_range + 1, width)):
            for b in range(max(int(y) - search_range, 0), min(int(y) + search_range + 1, height)):
                c = cells.get((a, b, int(p)))
                if c is not None:
                    diff = min(diff, np.min(np.abs(c - int(t))))
        if diff > cap:
            diff = cap
            overflow += 1
        total += diff
    return np.array([total / len(event_gt), overflow])


def _fields(ev):
    return tuple(np.asarray(ev[f]).astype(np.int64) for f in ('timestamp', 'x', 'y', 'polarity'))


def ts_diff_exact(gt, pred, search_range=0, fps=30, width=346, height=260):
    """(total, overflow) as integers: the sum of the distances at or below the cap and the number of capped events,
    i.e. result[0] and result[1] of v2ce_ts_diff_metric.  The metric is (total + overflow * cap) / len(gt)."""
    return totals(nearest_distances(gt, pred, search_range, width, height), fps)


def totals(best, fps, *, tie_overflows=False, clamp=True):
    """(total, overflow) from the per-event nearest distances: the distance is clamped to 1e6 and capped when it
    exceeds cap = 1e6/fps/10*3.  The switches make the errors of the mutation tests: tie_overflows counts a distance
    equal to the cap as overflow, clamp=False adds the unclamped distance (NONE for an empty window)."""
    cap = 1e6 / fps / 10 * 3
    d = np.minimum(best, 1000000)
    over = (d >= cap) if tie_overflows else (d > cap)
    if clamp:
        return int(d[~over].sum()), int(over.sum())
    return sum(int(v) for v in best[~over]), int(over.sum())


def nearest_distances(gt, pred, search_range=0, width=346, height=260, *, window_hi=1, swap_clamps=False,
                      polarity=True):
    """Per ground-truth event the smallest |t_pred - t_gt| (int64, NONE when the window holds no predicted event).
    The switches make the errors of the mutation tests: window_hi=0 ends the window one pixel short on the high side,
    swap_clamps clamps x by the height and y by the width, polarity=False ignores polarity."""
    return PredCells(pred, width, height, polarity).nearest(gt, search_range, window_hi, swap_clamps)


class PredCells:
    """The predicted events sorted by one int64 key, cell * 2^tb + (t - t_min) with cell = (x * height + y) * 2 + p,
    built once and queried with any ground-truth set and search range.  For every offset of the window the
    ground-truth keys of that neighbour cell are binary-searched; the predicted events on both sides of the insertion
    point that lie in the same cell are the nearest in time."""

    def __init__(self, pred, width=346, height=260, polarity=True):
        self.width, self.height, self.polarity = width, height, polarity
        tp, xp, yp, pp = _fields(pred)
        if not polarity:
            pp = np.where((pp == 0) | (pp == 1), 0, pp)
        # the only predicted events any window can reach: inside the sensor with polarity 0 / 1
        keep = (xp >= 0) & (xp < width) & (yp >= 0) & (yp < height) & ((pp == 0) | (pp == 1))
        tp, xp, yp, pp = tp[keep], xp[keep], yp[keep], pp[keep]
        self.n = len(tp)
        self.t0 = int(tp.min()) if self.n else 0
        self.tb = max(1, (int(tp.max()) - self.t0).bit_length()) if self.n else 1
        side = max(width, height) + 1
        if self.tb + (side * side * 2).bit_length() > 62:
            raise ValueError('PredCells: the time span does not fit the sort key next to the cell index')
        self.key = np.sort((((xp * height + yp) * 2 + pp) << self.tb) | (tp - self.t0))
        self.cell, self.t = self.key >> self.tb, (self.key & ((1 << self.tb) - 1)) + self.t0

    def nearest(self, gt, search_range=0, window_hi=1, swap_clamps=False):
        r, width, height = int(search_range), self.width, self.height
        tg, xg, yg, pg = _fields(gt)
        pg[pg == -1] = 0                                 # ground truth only, like the reference
        if not self.polarity:
            pg[:] = 0
        best = np.full(len(tg), NONE, dtype=np.int64)
        if not len(tg) or not self.n:
            return best
        # ground truth in (cell, t) order: shifting every cell by one constant keeps the queries sorted, which keeps
        # searchsorted cache-friendly; events far outside the sensor never reach a cell.  A query time outside the
        # predicted span is clipped into it, which still lands next to the first / last event of the cell.
        near = (xg >= -r) & (xg < width + r) & (yg >= -r) & (yg < height + r)
        idx = np.nonzero(near)[0]
        base = (xg[idx] * height + yg[idx]) * 2 + pg[idx]
        order = np.lexsort((tg[idx], base))
        idx, base = idx[order], base[order]
        gx, gy, gt_t = xg[idx], yg[idx], tg[idx]
        gdt = np.clip(gt_t - self.t0, 0, (1 << self.tb) - 1)
        sub = np.full(len(idx), NONE, dtype=np.int64)
        xlim, ylim = (height, width) if swap_clamps else (width, height)
        last = self.n - 1
        for dx in range(-r, r + window_hi):
            okx = (gx + dx >= 0) & (gx + dx < xlim)
            for dy in range(-r, r + window_hi):
                sel = np.nonzero(okx & (gy + dy >= 0) & (gy + dy < ylim))[0]
                if not len(sel):
                    continue
                qcell = base[sel] + (dx * height + dy) * 2
                at = np.searchsorted(self.key, (qcell << self.tb) | gdt[sel])
                for nb in (at - 1, at):
                    nbc = np.clip(nb, 0, last)
                    valid = (nb >= 0) & (nb <= last) & (self.cell[nbc] == qcell)
                    sub[sel] = np.minimum(sub[sel], np.where(valid, np.abs(self.t[nbc] - gt_t[sel]), NONE))
        best[idx] = sub
        return best


def _records(t, x, y, p):
    ev = np.zeros(len(t), dtype=np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')]))
    ev['timestamp'], ev['x'], ev['y'], ev['polarity'] = t, x, y, p
    return ev


def planted_edges(width, height, search_range, seed=0, t_base=0, n_background=0):
    """(gt, pred) whose answer shows which neighbour cells the window covered.  Ground-truth events sit on every
    corner, on the middle of every edge, one pixel inside and at the centre; each has one predicted event of its
    polarity at Chebyshev offset exactly r or r + 1 in one of the eight directions, at its own distance 1 + j (distinct
    for every group j), so a window that is one pixel too small or too large, or clamped by the wrong side, changes
    the total.  Every fourth group also has a predicted event of the other polarity at distance 0.  Groups are SEP
    apart in time; n_background random events of each kind are added over the whole sensor and time span."""
    rng = np.random.default_rng(seed)
    r = int(search_range)
    xs = sorted({v for v in (0, 1, width // 2, width - 2, width - 1) if 0 <= v < width})
    ys = sorted({v for v in (0, 1, height // 2, height - 2, height - 1) if 0 <= v < height})
    offs = sorted({(sx * k, sy * k) for k in (r, r + 1) for sx in (-1, 0, 1) for sy in (-1, 0, 1)
                   if (sx, sy) != (0, 0) or k == 0})
    g, q = [], []
    j = 0
    for x in xs:
        for y in ys:
            for ox, oy in offs:
                t = t_base + j * SEP
                p = int(rng.integers(0, 2))
                g.append((t, x, y, p))
                if 0 <= x + ox < width and 0 <= y + oy < height:
                    q.append((t + (1 + j) * (1 if j % 2 else -1), x + ox, y + oy, p))
                if j % 4 == 0:
                    q.append((t, x, y, 1 - p))
                j += 1
    g, q = np.array(g, dtype=np.int64).reshape(-1, 4), np.array(q, dtype=np.int64).reshape(-1, 4)
    if n_background:
        span = max(j, 1) * SEP
        bg = [np.column_stack([t_base + rng.integers(0, span, n_background), rng.integers(0, width, n_background),
                               rng.integers(0, height, n_background), rng.integers(0, 2, n_background)])
              for _ in range(2)]
        g, q = np.concatenate([g, bg[0]]), np.concatenate([q, bg[1]])
    return _records(*g.T), _records(*q.T)


def planted_distances(fps):
    """The distances where counting changes at this frame rate: 0, and the cap +- 1 while the cap is below 1e6;
    1e6 +- 1 and 2e6 (which the 1e6 clamp must turn into 1e6) once it is not."""
    cap = 1e6 / fps / 10 * 3
    if cap < 1e6:
        c = int(round(cap))
        return [0, c - 1, c, c + 1]
    return [0, 999999, 1000000, 1000001, 2000000]


def planted_times(fps, search_range, seed=0, t_base=0, repeat=4, n_empty=0, width=346, height=260):
    """(gt, pred) with ground-truth events whose nearest predicted event (same polarity, somewhere in the window) is
    exactly each of planted_distances(fps) away, before and after, `repeat` times each, and n_empty ground-truth
    events whose window holds no predicted event at all (in the right quarter of the sensor, which no predicted event
    enters).  Timestamps start at t_base."""
    rng = np.random.default_rng(seed)
    r = int(search_range)
    xmax = width - width // 4 - r          # windows of the planted groups stay left of the empty quarter
    g, q = [], []
    j = 0
    for d in planted_distances(fps):
        for k in range(2 * repeat):
            t = t_base + j * SEP
            x, y, p = int(rng.integers(0, max(xmax, 1))), int(rng.integers(0, height)), int(rng.integers(0, 2))
            ox, oy = (int(v) for v in rng.integers(-r, r + 1, 2))
            g.append((t, x, y, p))
            q.append((t + (d if k % 2 else -d), min(max(x + ox, 0), width - 1), min(max(y + oy, 0), height - 1), p))
            j += 1
    for _ in range(n_empty):
        g.append((t_base + j * SEP, int(rng.integers(xmax + r + r, width)), int(rng.integers(0, height)),
                  int(rng.integers(0, 2))))
        j += 1
    g, q = np.array(g, dtype=np.int64).reshape(-1, 4), np.array(q, dtype=np.int64).reshape(-1, 4)
    return _records(*g.T), _records(*q.T)
