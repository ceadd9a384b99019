"""Host side of LDATI (stage 2): constants, workspaces and the two-phase C-ABI calls.

Mirrors what /root/reference/scripts/LDATI.py:126-214 does on the host (shape checks,
scalar constants) and hands all tensor work to libv2ce_b200.so:

    v2ce_ldati_count  -> per-(frame,bin) event counts              (LDATI.py:80-106)
    [one small D2H: the counts size the output, as `torch.max(y)` does at LDATI.py:169]
    v2ce_ldati_emit   -> timestamps, stable segment sort, 13-byte records (LDATI.py:156-310)
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from ._lib import LdatiParams, V2ceError, check, ptr, stream_ptr

EVENT_DTYPE = np.dtype([('timestamp', '<i8'), ('x', '<i2'), ('y', '<i2'), ('polarity', 'i1')])
NBINS = 9
KEY_BIAS = 8
STRATEGIES = {'none': 0, 'slope': 1, 'random': 2}     # v2ce_ldati_params.multi_events
POOLING = {'none': 0, 'weighted': 1, 'avg': 2}        # v2ce_ldati_params.pooling
BIDIR_MAX_TENDENCY = 1024                             # largest tenth-bin voxel value the bidirectional sort window accepts


_bin_starts_cache = {}


def bin_starts(fps, device, flavor='cuda'):
    """Cached per (fps, device, flavour): evaluating it reads a device tensor back, i.e. synchronises the
    current stream, which a pipelined caller (runner.BatchRunner) must not do per batch."""
    key = (fps, str(device), flavor)
    if key not in _bin_starts_cache:
        _bin_starts_cache[key] = _bin_starts(fps, device, flavor)
    return _bin_starts_cache[key]


def _bin_starts(fps, device, flavor='cuda'):
    """`torch.arange(0, frame_step, voxel_step)` exactly as the reference evaluates it
    (LDATI.py:164,209): on the CUDA device for the torch-CUDA flavour, on CPU otherwise."""
    frame_step = 1 / fps
    voxel_step = 1 / fps / NBINS
    dev = device if flavor == 'cuda' else 'cpu'
    return torch.arange(0, frame_step, voxel_step, device=dev).cpu().numpy().astype(np.float32)


def make_params(n_frames, height, width, fps=30, t0=0, seed=0, frame_base=0, flavor='cuda',
                device='cuda', add_frame_offset=False, additional_events_strategy='slope', bidirectional=False,
                pooling_type='none', pooling_kernel_size=3):
    """Scalar constants with the reference's own Python expressions (SURVEY.md Appendix A)."""
    if additional_events_strategy not in STRATEGIES:
        raise ValueError(f'additional_events_strategy must be one of {sorted(STRATEGIES)}')
    assert flavor in ('cuda', 'cpu')
    f32 = np.float32
    voxel_step = 1 / fps / NBINS                       # LDATI.py:146
    p = LdatiParams()
    p.height, p.width, p.n_frames = height, width, n_frames
    p.true_div = 1 if flavor == 'cpu' else 0
    p.frame_base = frame_base
    p.seed = seed & 0xFFFFFFFFFFFFFFFF
    p.fps64, p.nbins64 = float(fps), float(NBINS)
    p.r_fps64, p.r_nbins64 = 1.0 / fps, 1.0 / NBINS
    p.fps32, p.nbins32 = f32(fps), f32(NBINS)
    p.r_fps32, p.r_nbins32 = f32(1.0 / fps), f32(1.0 / NBINS)
    p.vs32 = f32(voxel_step)
    p.inv_vs32 = f32(1 / voxel_step)
    p.vs2_32 = f32(voxel_step ** 2)
    p.r_vs2_32 = f32(1.0 / (voxel_step ** 2))
    p.six32, p.r6_32 = f32(6), f32(1.0 / 6)
    p.eps6, p.eps8 = f32(1e-6), f32(1e-8)
    bs = bin_starts(fps, device, flavor)
    if bs.shape[0] != NBINS:
        raise V2ceError(f'torch.arange(0, 1/{fps}, 1/{fps}/9) has {bs.shape[0]} entries; the reference '
                        f'would fail to broadcast it against 9 bins')
    bs_t0 = (bs + f32(t0)).astype(f32)                 # `arange + t0` is a float32 add
    # Sort-key window per bin: the key of an event is ts - bin_base_us + KEY_BIAS and must land in [1, 2^key_bits).
    one_bin = int(math.ceil(1e6 / fps / NBINS))
    below, span = 0, one_bin + 2                       # 'slope' / 'none': offsets in [0, voxel_step]
    if bidirectional:
        # bin 5's tendency is bless - debt > -1 bin (LDATI.py:121); bin 8's is the tenth voxel bin itself
        # (LDATI.py:108,111), accepted up to BIDIR_MAX_TENDENCY bins -- beyond it the emit status flags the event
        below = one_bin + 2
        span = BIDIR_MAX_TENDENCY * one_bin + 2
    if additional_events_strategy == 'random':
        span = max(span, 1_000_000 + 64)               # the raw draw in [0, 1) is taken as seconds (LDATI.py:173-174)
    for c in range(NBINS):
        p.binstart_t0_32[c] = bs_t0[c]
        p.bin_base_us[c] = int(math.floor(float(bs_t0[c]) * 1e6)) - below
    p.key_span = below + span + 2 * KEY_BIAS
    p.add_frame_offset = 1 if add_frame_offset else 0
    p.multi_events = STRATEGIES[additional_events_strategy]
    p.bidirectional = 1 if bidirectional else 0
    if pooling_type not in POOLING:
        raise ValueError(f'pooling_type must be one of {sorted(POOLING)}')
    if pooling_type == 'avg' and pooling_kernel_size % 2 == 0:
        raise ValueError('pooling_kernel_size must be odd: an even AvgPool2d kernel changes the plane size '
                         '(the reference fails in its reshape, LDATI.py:186)')
    # only the 'slope' strategy reads the pooled counts (LDATI.py:175-183)
    p.pooling = POOLING[pooling_type] if additional_events_strategy == 'slope' else 0
    p.pooling_kernel_size = int(pooling_kernel_size)
    return p


class LdatiEngine:
    """Reusable workspaces + the count / emit calls for one device."""

    def __init__(self, device='cuda'):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self._count_ws = None
        self._emit_ws = None
        self.launches = 0

    def _ws(self, attr, nbytes):
        buf = getattr(self, attr)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.device)
            setattr(self, attr, buf)
        return buf

    def count(self, voxels, params, out=None, ef_sums=None):
        """voxels (F,2,10,H,W) float32 CUDA contiguous -> seg_counts int64 (F,9) on device (`out` if given).
        ef_sums: optional float32 (F,2,H,W) CUDA tensor that receives the per-polarity event-frame sums
        (event_frames.accumulate(keep_polarity=True)) from the same read of the voxels."""
        n = ctypes.c_size_t()
        check(self.lib.v2ce_ldati_count_workspace_bytes(ctypes.byref(params), ctypes.byref(n)))
        ws = self._ws('_count_ws', n.value)
        seg = out if out is not None else torch.empty((params.n_frames, NBINS), dtype=torch.int64, device=self.device)
        check(self.lib.v2ce_ldati_count_ef(ptr(voxels), ctypes.byref(params), ptr(ws), ws.numel(), ptr(seg),
                                           ptr(ef_sums), stream_ptr()))
        self.launches += 3
        return seg

    def emit(self, voxels, params, total_events, draws=None, frame_offsets=None, out=None, status_out=None):
        """Second phase.  Returns (events uint8 (total*13,) on device, status int32[4] on device)."""
        n = ctypes.c_size_t()
        check(self.lib.v2ce_ldati_emit_workspace_bytes(ctypes.byref(params), total_events, ctypes.byref(n)))
        ws = self._ws('_emit_ws', n.value)
        if out is None:
            out = torch.empty(max(total_events, 1) * EVENT_DTYPE.itemsize, dtype=torch.uint8, device=self.device)
        status = status_out if status_out is not None else torch.empty(4, dtype=torch.int32, device=self.device)
        m = 0
        if draws is not None:
            m = draws.shape[-1]
        check(self.lib.v2ce_ldati_emit(ptr(voxels), ctypes.byref(params), ptr(self._count_ws), ptr(ws), ws.numel(),
                                       ptr(draws), m, ptr(frame_offsets), total_events, ptr(out), ptr(status),
                                       stream_ptr()))
        key_bits = max(1, math.ceil(math.log2(params.key_span + 1)))
        passes = (key_bits + 5) // 6                 # one-sweep passes of <= 6 bits (csrc/ldati.cu, osw_*)
        # emit + tile table (build, fill) + digit histograms + one kernel per pass + pack (chunk table, records)
        self.launches += 1 + (2 + 1 + passes + 2 if total_events > 0 else 0)
        return out, status

    def run(self, voxels, params, draws=None, frame_offsets=None):
        """count -> (sync on the segment counts) -> emit.  Returns (events_dev, seg_counts_host)."""
        seg = self.count(voxels, params)
        seg_host = seg.cpu().numpy()
        total = int(seg_host.sum())
        events, status = self.emit(voxels, params, total, draws, frame_offsets)
        return events, seg_host, status


_engines = {}


def engine_for(device):
    device = torch.device(device)
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _engines:
        _engines[key] = LdatiEngine(device)
    return _engines[key]


def frame_offsets_us(pair_base, n, fps):
    """int64 (n,): the per-frame timestamp offsets `int(i * 1 / fps * 1e6)` of v2ce.py:365 for i = pair_base ..
    pair_base+n-1 -- Python's int/int true division is the correctly rounded quotient, which for |i|, fps < 2^53 is the
    float64 division numpy does; then one float64 multiply and a truncation."""
    i = np.arange(pair_base, pair_base + n, dtype=np.int64).astype(np.float64)
    return (i / np.float64(fps) * np.float64(1e6)).astype(np.int64)


def check_status(status_host):
    if int(status_host[0]) != 0:
        raise V2ceError(f'LDATI: {int(status_host[0])} timestamps fell outside the sort-key range '
                        f'(non-finite or out-of-contract voxel values)')


def records_dev(ev, device):
    """Packed 13-byte records on `device` and their count.  `ev`: a uint8 CUDA tensor of packed records (used as it
    is) or a host record array with the fields timestamp, x, y, polarity of any integer widths (converted to
    EVENT_DTYPE, then uploaded)."""
    if isinstance(ev, torch.Tensor):
        if not ev.is_cuda or ev.dtype != torch.uint8 or ev.numel() % 13:
            raise V2ceError('event tensors must be uint8 CUDA tensors of packed 13-byte records')
        return ev.contiguous().reshape(-1), ev.numel() // 13
    ev = np.asarray(ev)
    if ev.dtype != EVENT_DTYPE:
        rec = np.empty(ev.shape[0], dtype=EVENT_DTYPE)
        for f in ('timestamp', 'x', 'y', 'polarity'):
            rec[f] = ev[f]
        ev = rec
    flat = torch.from_numpy(np.ascontiguousarray(ev).view(np.uint8).reshape(-1))
    return flat.to(device), ev.shape[0]


def split_frames(events_host, seg_counts_host):
    """events_host: uint8 (total*13,) host array -> list of per-frame recarrays (views)."""
    rec = events_host.view(EVENT_DTYPE)
    per_frame = seg_counts_host.sum(axis=1)
    out, start = [], 0
    for n in per_frame:
        out.append(rec[start:start + int(n)].view(np.recarray))
        start += int(n)
    return out
