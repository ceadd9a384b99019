"""Event stream -> voxel grid on libv2ce_b200.so (csrc/voxelize.cu): the step between a ground-truth recording and the
stage-2 samplers (sample_voxel_statistical, sample_voxel_baseline), kept on the device.

    events_to_voxels(events, n_frames=None, fps=30, *, t0_us=0, frame_edges_us=None, nbins=10, width=346, height=260,
                     device=None) -> torch.Tensor     # float32 (F, 2, nbins, H, W) on the device

This is the toolbox's own binning convention.  It is NOT a port of the reference's training voxeliser
(train/scripts/utils/events_utils.py), and no parity with it is claimed.  Per event:

  1. x outside [0, width) or y outside [0, height): IndexError (like ts_diff_metric);
  2. polarity 1 -> plane 0, polarity 0 or -1 -> plane 1 (LDATI's plane order; ts_diff_metric treats -1 as 0);
     any other value: ValueError;
  3. t < e[0] or t >= e[F]: dropped (the normal case when voxelising part of a recording);
  4. frame f with e[f] <= t < e[f+1], L = e[f+1] - e[f], r = t - e[f]; bin c = ((r + 1) * nbins - 1) // L in exact
     int64, i.e. bin c starts at e[f] + floor(c * L / nbins).  Floor-rounded starts match the samplers, which truncate
     their timestamps: the first event they place in bin c sits at a floor-rounded microsecond;
  5. voxels[f, plane, c, y, x] += 1.

The counts are exact while a cell stays below 2^24 events, and then do not depend on the order of the events.

Frame edges (int64 us): by default e[f] = t0_us + int(f / fps * 1e6), f = 0..n_frames -- the CLI's own per-frame
offsets (v2ce.py:365, ldati.frame_offsets_us), so the stream the CLI writes lands back in the frames it came from, bar
events a sampler placed at or after the next frame's start.  Recordings with measured frame times pass
``frame_edges_us`` (F + 1 strictly increasing values) instead of ``n_frames``.

``events``: a host record array with the fields timestamp, x, y, polarity (any integer widths), or a uint8 CUDA tensor
of packed 13-byte records (e.g. ``stream_clip(..., events_to_host=False).event_stream_dev``).  There is no CPU path."""
import numpy as np
import torch

from . import _lib
from ._lib import V2ceError, check, ptr, stream_ptr
from .ldati import EVENT_DTYPE, frame_offsets_us, records_dev


def _frame_edges(n_frames, fps, t0_us, frame_edges_us, nbins):
    if (n_frames is None) == (frame_edges_us is None):
        raise ValueError('events_to_voxels: pass exactly one of n_frames and frame_edges_us')
    if frame_edges_us is None:
        if int(n_frames) != n_frames or n_frames < 1:
            raise ValueError(f'events_to_voxels: n_frames must be a positive integer, got {n_frames}')
        if not fps > 0:
            raise ValueError(f'events_to_voxels: fps must be positive, got {fps}')
        edges = frame_offsets_us(0, int(n_frames) + 1, fps) + np.int64(t0_us)
    else:
        edges = np.asarray(frame_edges_us)
        if edges.ndim != 1 or edges.shape[0] < 2 or not np.issubdtype(edges.dtype, np.integer):
            raise ValueError('events_to_voxels: frame_edges_us must be a 1-D integer array of F + 1 >= 2 edges')
        edges = edges.astype(np.int64)
    if not (edges[1:] > edges[:-1]).all():
        raise ValueError('events_to_voxels: the frame edges must be strictly increasing')
    longest = max(int(b) - int(a) for a, b in zip(edges[:-1].tolist(), edges[1:].tolist()))
    if longest * nbins >= 1 << 62:
        raise ValueError(f'events_to_voxels: a frame of {longest} us x {nbins} bins does not fit the int64 bin arithmetic')
    return edges


def _check_field_ranges(events, width, height):
    """Host records wider than the packed fields: a value the packed field cannot hold would wrap on conversion."""
    if isinstance(events, torch.Tensor):
        return
    ev = np.asarray(events)
    if ev.dtype == EVENT_DTYPE or ev.shape[0] == 0:
        return
    for f, lim in (('x', width), ('y', height)):
        if not np.can_cast(ev.dtype[f], EVENT_DTYPE[f]):
            a = ev[f]
            if a.min() < 0 or a.max() >= lim:
                raise IndexError(f'events_to_voxels: events outside the {width}x{height} sensor')
    if not np.can_cast(ev.dtype['polarity'], EVENT_DTYPE['polarity']):
        a = ev['polarity']
        if a.min() < -1 or a.max() > 1:
            raise ValueError('events_to_voxels: polarity values other than -1, 0 and 1')


def events_to_voxels(events, n_frames=None, fps=30, *, t0_us=0, frame_edges_us=None, nbins=10, width=346, height=260,
                     device=None) -> torch.Tensor:
    if device is None:
        device = events.device if isinstance(events, torch.Tensor) else 'cuda'
    device = torch.device(device)
    if device.type != 'cuda':
        raise V2ceError('events_to_voxels (B200) has no CPU path')
    if int(nbins) != nbins or nbins < 1:
        raise ValueError(f'events_to_voxels: nbins must be a positive integer, got {nbins}')
    if width < 1 or height < 1:
        raise ValueError(f'events_to_voxels: bad sensor {width}x{height}')
    edges = _frame_edges(n_frames, fps, t0_us, frame_edges_us, int(nbins))
    _check_field_ranges(events, width, height)
    F = edges.shape[0] - 1
    lib = _lib.load()
    with torch.cuda.device(device):
        rec, n = records_dev(events, device)
        edges_dev = torch.from_numpy(edges).to(device)
        vox = torch.empty((F, 2, int(nbins), height, width), dtype=torch.float32, device=device)
        status = torch.empty(4, dtype=torch.int64, device=device)
        check(lib.v2ce_events_to_voxels(ptr(rec), n, ptr(edges_dev), F, int(nbins), height, width, ptr(vox), ptr(status),
                                        stream_ptr()))
        outside, bad_polarity, _, _ = (int(v) for v in status.cpu().tolist())
    if outside:
        raise IndexError(f'events_to_voxels: {outside} events outside the {width}x{height} sensor')
    if bad_polarity:
        raise ValueError(f'events_to_voxels: {bad_polarity} events with a polarity other than -1, 0 and 1')
    return vox
