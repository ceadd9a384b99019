"""ClipStream: convert frames to events as they arrive, from host or CUDA frames, gray or colour.

    with ClipStream(model, fps=30, seq_len=16, batch_size=4, seed=0, color='rgb') as cs:
        for frames in source:                     # uint8 (n, H, W) gray or (n, H, W, C) colour; ndarray or CUDA tensor
            for b in cs.push(frames):             # zero or more finished batches
                consume(b.events_dev, b.pair_range)
        res = cs.close()                          # the last batches, preview frames, upper bound, pair count

For the same frames, model state and arguments, the concatenated events of all batches, ``res.ef_frames``,
``res.ef_upper_bound`` and ``res.n_pairs`` are byte-identical to ``v2ce.stream_clip`` on those frames, however the
frames are split across ``push`` calls.  That holds because the reference's window schedule (v2ce.py:149-154) changes
only at the end of a clip: window k starts at k * seq_len and is final once its seq_len + 1 frames exist, and only the
last window can be pulled back.  So batch j (windows j*b .. j*b+b-1, the model calls of ``stream_clip`` in the same
order) is submitted as soon as frame (j+1)*b*seq_len exists, and the batch holding the last window at ``close()``.

Frames reach the model through one kernel, ``frames.assemble_windows``: it builds a batch's uint8 gray windows from
the frames where they lie, converting colour as cv2.cvtColor(*2GRAY) does (the reference's video reader,
scripts/video_reader.py:66-67), center-cropped for the native route and whole for the resize / pano route
(v2ce._frame_route, the rule ``stream_clip`` uses).  Host frames are copied when pushed and uploaded one by one when a
batch first needs them; CUDA frames are read in place, so a pushed CUDA tensor must not be written to until the stream
no longer holds it (at most (batch_size + 1) * seq_len frames after it).

Memory stays bounded: the stream holds only the frames that a batch not yet submitted may read, each batch's events are
handed out and not kept, and the only state that grows with the clip is the per-pair event-frame sums of the
clip-global percentile (v2ce.py:262-264), 2 * H * W float32 per pair (0.72 MB at 346 x 260), none with
write_event_frames=False.  A handed-out batch owns its events: they are copied out of the runner's slot on the copy
stream, the same device-to-device copy (13 bytes per event read and written) ``stream_clip`` makes into its clip-wide
buffer.
"""
import numpy as np
import torch

from . import frames as _frames
from . import v2ce as _drv


class StreamSchedule:
    """The batches a stream of frames is cut into: ``add(n)`` returns those that n more frames complete, ``finish()``
    the rest once the clip's length is known, each as (frame index ranges of its windows, trim_last_window_to).  The
    windows are v2ce.window_schedule's and the batches v2ce.batch_plan's, for any way the frames arrive."""

    def __init__(self, seq_len, batch_size):
        if seq_len < 1 or batch_size < 1:
            raise ValueError(f'seq_len and batch_size must be >= 1, got {seq_len}, {batch_size}')
        self.seq_len, self.batch_size = seq_len, batch_size
        self.n_frames = 0
        self.n_batches = 0                      # batches returned so far

    def add(self, n):
        self.n_frames += n
        L, b = self.seq_len, self.batch_size
        out = []
        # batch j's last window, (j+1)*b - 1, is final once frame (j+1)*b*L exists; no later pull-back can move it
        while self.n_frames >= (self.n_batches + 1) * b * L + 1:
            k0 = self.n_batches * b
            out.append(([range(k * L, k * L + L + 1) for k in range(k0, k0 + b)], 0))
            self.n_batches += 1
        return out

    def finish(self):
        L = self.seq_len
        starts, mode = _drv.window_schedule(self.n_frames, L)
        plan = _drv.batch_plan(starts, mode, self.batch_size)
        # a clip of <= seq_len frames has a negative start; range slicing clamps it like the image list of v2ce.py:158-166
        frames = range(self.n_frames)
        out = [([frames[int(s):int(s) + L + 1] for s in starts[a:e]], trim) for a, e, trim in plan[self.n_batches:]]
        self.n_batches = len(plan)
        return out

    @property
    def keep_from(self):
        """First frame a batch not yet returned may read: a pulled-back last window starts after its predecessor."""
        return max(0, (self.n_batches * self.batch_size - 1) * self.seq_len + 1)


class StreamBatch:
    """One batch of a ClipStream: packed 13-byte event records (timestamps absolute, v2ce.py:365) of the frame pairs
    [pair_range[0], pair_range[1]) in a uint8 CUDA tensor of its own."""

    def __init__(self, events_dev, pair_range):
        self.events_dev = events_dev
        self.pair_range = pair_range
        self.n_events = events_dev.numel() // 13


class StreamResult:
    def __init__(self, batches, ef_frames, ef_upper_bound, n_pairs):
        self.batches = batches                  # the batches close() handed out
        self.ef_frames = ef_frames              # uint8 BGR (n_pairs, H, W, 3) | None, like ClipResult.ef_frames
        self.ef_upper_bound = ef_upper_bound
        self.n_pairs = n_pairs


class ClipStream:
    def __init__(self, model, fps=30, seq_len=16, width=346, height=260, infer_type='center', batch_size=4, seed=0,
                 pair_base=0, ceil=10, upper_bound_percentile=98, keep_polarity=True, write_event_frames=True,
                 color='gray', device=None):
        if color not in _frames.COLORS:
            raise ValueError(f'color must be one of {sorted(_frames.COLORS)}, got {color!r}')
        if infer_type not in ('center', 'pano'):
            raise ValueError(f'infer_type must be center or pano, got {infer_type!r}')
        self.schedule = StreamSchedule(seq_len, batch_size)
        _drv._claim_model(model)
        self.model, self.color, self.infer_type = model, color, infer_type
        self.fps, self.seed, self.pair_base, self.ceil, self.percentile = fps, seed, pair_base, ceil, upper_bound_percentile
        self.keep_polarity, self.write_event_frames = keep_polarity, write_event_frames
        self.width, self.height = width, height
        self.device = torch.device(device or 'cuda')
        self._ring = {}                         # frame index -> uint8 CUDA tensor (H, W[, C])
        self._shape = None                      # of one frame
        self._route = None
        self._clip = None                       # v2ce._ClipRun, from the first batch on
        self._prev = None                       # ticket submitted last: handed out after the next submit, or by close()
        self._closed = False

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if not self._closed:                    # left without close(): give the model back, hand out nothing
            self._closed = True
            _drv._release_model(self.model)
        return False

    # ------------------------------------------------------------------------------------------
    def push(self, frames):
        """Add frames, uint8 (n, H, W) gray or (n, H, W, C) colour in this stream's colour order, host ndarray or CUDA
        tensor.  Returns the batches (StreamBatch) whose events are complete, in order; possibly none."""
        if self._closed:
            raise RuntimeError('push() after close()')
        views = self._check(frames)
        out = []
        for f in views:                         # frame by frame: one push of a whole clip keeps the ring as small
            self._ring[self.schedule.n_frames] = f
            for windows, trim in self.schedule.add(1):
                out += self._run(windows, trim)
            for i in [i for i in self._ring if i < self.schedule.keep_from]:
                del self._ring[i]
        return out

    def close(self):
        """End of the clip: submits the batch holding the last window and returns a StreamResult with the batches not
        handed out yet, the preview frames, their upper bound and the pair count.  Fails as stream_clip fails on the same
        frames given as an image list (a clip of seq_len frames has a one-frame window)."""
        if self._closed:
            raise RuntimeError('close() was called already')
        self._closed = True
        try:
            out = []
            for windows, trim in self.schedule.finish():
                out += self._run(windows, trim)
            if self._prev is None:              # a clip of at most one frame: no window (stream_clip's empty result)
                return StreamResult(out, None, None, 0)
            with torch.cuda.device(self.device):
                out += self._hand_out(self._prev)
                self._prev = None
                frames, ub, _ = self._clip.event_frames(self.write_event_frames)
            return StreamResult(out, frames, ub, self._clip.pair_idx - self.pair_base)
        finally:
            self._ring.clear()
            _drv._release_model(self.model)

    # ------------------------------------------------------------------------------------------
    def _check(self, frames):
        c = _frames.COLORS[self.color][0]
        if isinstance(frames, torch.Tensor):
            if frames.dtype != torch.uint8:
                raise ValueError(f'frames must be uint8, got {frames.dtype}')
            if not frames.is_cuda:
                frames = frames.numpy()
        else:
            frames = np.asarray(frames)
            if frames.dtype != np.uint8:
                raise ValueError(f'frames must be uint8, got {frames.dtype}')
        want = 3 if c == 1 else 4
        if frames.ndim != want or (c > 1 and frames.shape[-1] != c):
            raise ValueError(f'{self.color} frames are (n, ' + ', '.join(['H', 'W'] + ([str(c)] if c > 1 else [])) +
                             f'), got {tuple(frames.shape)}')
        shape = tuple(frames.shape[1:])
        if self._shape is None:
            route, _ = _drv._frame_route(self.model, self.infer_type, np.uint8, (1,) + shape[:2], self.height,
                                         self.width, True)
            if route is None:
                raise ValueError(f'frames of {shape[0]} x {shape[1]} pixels cannot be converted (fewer than 2 rows)')
            self._shape, self._route = shape, route
        elif shape != self._shape:
            raise ValueError(f'frames of shape {shape} after frames of shape {self._shape}')
        if isinstance(frames, torch.Tensor):
            dev = self.device if self.device.index is not None else torch.device('cuda', torch.cuda.current_device())
            if frames.device != dev:
                raise ValueError(f'frames on {frames.device}, the stream runs on {dev}')
            return [_frames.device_frame(f, self.color) for f in frames]
        return [_HostFrame(f) for f in frames]

    def _device_frame(self, f):
        if isinstance(f, _HostFrame):           # uploaded when a batch first needs it, then kept as a device frame
            f = f.upload(self.device)
        return f

    def _run(self, windows, trim):
        """Assemble one batch's windows on the device, submit it, and hand out the batch submitted before it."""
        with torch.cuda.device(self.device):
            src = sorted({i for w in windows for i in w})
            for i in src:
                self._ring[i] = self._device_frame(self._ring[i])
            pos = {i: j for j, i in enumerate(src)}
            slots = np.array([[pos[i] for i in w] for w in windows], np.int32)
            H, W = self._shape[:2]
            x0, w_out = (W // 2 - self.width // 2, self.width) if self._route == 'native' else (0, W)
            x = _frames.assemble_windows([self._ring[i] for i in src], slots, self.color, x0, w_out)
            if self._clip is None:
                _, infer = _drv._frame_route(self.model, self.infer_type, np.uint8, (1, H, W), self.height, self.width,
                                             True)
                self._clip = _drv._ClipRun(self.model, self.device, infer, self.fps, self.ceil, self.percentile,
                                           self.keep_polarity, self.seed, self.pair_base,
                                           keep_sums=self.write_event_frames, hand_out=True)
            t = self._clip.submit(x, trim)
            out = self._hand_out(self._prev) if self._prev is not None else []
            self._prev = t
            return out

    def _hand_out(self, t):
        self._clip.runner.wait(t)               # status check; the copy of its events has finished
        ev = t.events_out
        ev.record_stream(torch.cuda.current_stream())   # allocated on the copy stream, used on the caller's
        return [StreamBatch(ev, (t.pair_base, t.pair_base + t.n_pairs))]


class _HostFrame:
    """A host frame waiting in the ring: a copy, so the caller may reuse its buffer as soon as push() returns."""

    def __init__(self, a):
        self.a = np.array(a, copy=True)

    def upload(self, device):
        return torch.from_numpy(self.a).pin_memory().to(device, non_blocking=True)
