"""BatchRunner: the hot path for one batch of windows, software-pipelined over three CUDA streams.

    image units (pinned host or device) ─H2D→ V2ce3d ─→ voxels ─→ event-frame sums, order statistics
                                                         └─→ LDATI count ─(counts D2H)→ emit/sort/pack ─D2H→ host events

The conv kernels of V2ce3d are persistent CTAs that leave most of an SM's registers, threads and HBM
bandwidth unused, while event frames and LDATI are short bandwidth/latency-bound launches with one
data-dependent host read in the middle (the counts size the output, as ``torch.max(y)`` does at
LDATI.py:169).  Run back to back they cost 1.1 ms of an 11.3 ms step and leave the GPU idle during the host
read.  Here they run on a second stream, one batch behind the network:

    submit(i):  main stream   UNet(i)                                   (enqueued first, asynchronously)
                host          wait for counts / order statistics of batch i-1   (the GPU is busy with UNet(i))
                post stream   stage B(i-1): event-frame normalise, LDATI emit/sort/pack
                copy stream   D2H of events / frames of batch i-1
                post stream   stage A(i):   after UNet(i): event-frame sums + radix select, LDATI count, small D2H

``wait(t)`` flushes stage B of ``t`` if no later submit has done so.  Buffers are per slot (``slots`` >= 2), so
``submit`` may be called for batch i+1 before ``wait`` is called for batch i.  ``bench.py`` (value and e2e)
and the tests drive it; it composes the same C-ABI calls as the one-by-one public functions
(``V2ce3d.__call__``, ``event_frames.*``, ``LdatiEngine.count/emit``).
"""
import contextlib
import ctypes
import os

import numpy as np
import torch

from . import _lib
from . import event_frames as _ef
from . import ldati as _ldati
from ._lib import check, ptr, stream_ptr


_NVTX = os.environ.get('V2CE_NVTX', '0') not in ('', '0')


@contextlib.contextmanager
def nvtx(name):
    """NVTX range around a pipeline stage (V2CE_NVTX=1; `ncu --nvtx --nvtx-include "v2ce:unet/"` then profiles one stage)."""
    if not _NVTX:
        yield
        return
    torch.cuda.nvtx.range_push(name)
    try:
        yield
    finally:
        torch.cuda.nvtx.range_pop()


class Ticket:
    __slots__ = ('slot', 'n_pairs', 'total', 'seg_counts', 'done', 'status', 'ub', 'h2d_bytes', 'd2h_bytes', 'hw',
                 'pair_base', 'vox', 'sums', 'small_host', 'counts_ready', 'staged', 'params', 'offs', 'fwd_events',
                 'events_dev', 'frames_dev', 'packed', 'ev_host')


class BatchRunner:
    def __init__(self, model, device, fps=30, ceil=10, percentile=98, keep_polarity=True, seed=0,
                 per_batch_frames=True, slots=3, copy_out=True, infer=None, collect_on_device=False):
        self.model = model
        self.device = torch.device(device)
        self.fps, self.ceil, self.percentile, self.keep = fps, ceil, percentile, keep_polarity
        self.seed = seed
        self.per_batch_frames = per_batch_frames
        self.copy_out = copy_out                  # False: results stay on the device (device-timed bench)
        # x on the device -> (b,L,20,H,W) voxels; default: the model itself (raw uint8 windows go through forward_frames).
        # v2ce.stream_clip passes the reference's center-crop / pano-tile wrappers (v2ce.py:66-129).
        self.infer = infer
        # True: the packed events of every batch are appended to one growing device buffer (copy stream) and read
        # back once by collected_events(): one D2H and one host array for a whole clip instead of a staging copy,
        # a pageable copy and a concatenation per batch (v2ce.stream_clip)
        self.collect_on_device = collect_on_device
        # multi-GPU e2e: an object whose place(slot, nbytes) returns the pinned host bytes this batch's events go to
        # (dist.SharedHostRing: this rank's slice of a shared-memory array that holds the merged stream of all ranks)
        self.host_sink = None
        self._all_ev = None
        self._all_bytes = 0
        self.clip_pairs = 0                     # pairs of the clip being collected (v2ce.stream_clip sets it): sizes
        self._pairs_collected = 0               # the clip-wide buffer after the first batch instead of regrowing it
        self.lib = _lib.load()
        # the network runs on its own HIGH-priority stream: the conv kernels are single-wave persistent CTAs that need a
        # whole SM's shared memory, so a CTA that has to wait for a post-stream block to leave its SM delays its whole
        # share of the tiles; with priority its CTAs are placed first (step 9.59 -> 9.44 ms on one box, DESIGN.md 4.7).
        # V2CE_NET_STREAM=0: the caller's current stream, as before.
        self.net_stream = torch.cuda.Stream(device=self.device, priority=-1) \
            if os.environ.get('V2CE_NET_STREAM', '1') not in ('', '0') else None
        self.post_stream = torch.cuda.Stream(device=self.device)      # event frames + LDATI, one batch behind
        self.copy_stream = torch.cuda.Stream(device=self.device)      # D2H of results
        self.h2d_stream = torch.cuda.Stream(device=self.device)       # H2D of inputs (PCIe is full duplex)
        self.slots = slots
        self.engines = [_ldati.LdatiEngine(self.device) for _ in range(slots)]    # count workspace per slot
        self._ev_dev = [None] * slots
        self._ev_host = [None] * slots
        self._fr_dev = [None] * slots
        self._fr_host = [None] * slots
        self._x_dev = [None] * slots
        self._sel_ws = [None] * slots
        self._small_dev = [None] * slots
        self._st_dev = [None] * slots
        self._small_host = [None] * slots
        self._offs_host = [None] * slots
        self._offs_dev = [None] * slots
        self._st_host = [torch.empty(4, dtype=torch.int32, pin_memory=True) for _ in range(slots)]
        self._free = [None] * slots            # event: every stream has finished with the slot's buffers
        self._next = 0
        self._pending = None                   # ticket whose stage B has not been enqueued yet
        self.launches = 0
        self.time_forward = False              # True: CUDA events around every forward (bench roofline)
        self.sums = []                         # per-batch event-frame sums (kept for a clip-global percentile)

    def _buf(self, lst, slot, nbytes, pinned=False):
        b = lst[slot]
        if b is None or b.numel() < nbytes:
            n = (int(nbytes * 1.25) + 256 + 63) // 64 * 64
            b = torch.empty(n, dtype=torch.uint8, pin_memory=True) if pinned else \
                torch.empty(n, dtype=torch.uint8, device=self.device)
            lst[slot] = b
        return b

    # ------------------------------------------------------------------------------------------
    def submit(self, units, pair_base, keep_sums=False, trim_last_window_to=0):
        """units: image units (b,L,2,H,W) float32, or raw gray windows (b,L+1,H,W) uint8 at the model's resolution;
        pinned host (copied on the side stream) or already on the device.  trim_last_window_to = m > 0: only the last m
        pairs of the batch's last window are kept (the clip's pulled-back last window, v2ce.py:227-236)."""
        t = Ticket()
        slot = self._next
        self._next = (self._next + 1) % self.slots
        t.slot, t.pair_base = slot, pair_base
        t.staged = False
        caller = torch.cuda.current_stream(self.device)
        cur = self.net_stream if self.net_stream is not None else caller
        if cur is not caller:
            cur.wait_stream(caller)               # device inputs were produced on the caller's stream
            if units.is_cuda:
                units.record_stream(cur)
        if self._free[slot] is not None:
            # the previous user of this slot has left the device: its per-slot pinned staging (counts, frame offsets)
            # is about to be rewritten by the host, its device buffers by this batch
            self._free[slot].synchronize()
            cur.wait_event(self._free[slot])
        t.h2d_bytes = 0
        if not units.is_cuda:
            t.h2d_bytes = units.numel() * units.element_size()
            with torch.cuda.stream(self.h2d_stream):
                x = units.to(self.device, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(self.h2d_stream)
            cur.wait_event(ready)
            x.record_stream(cur)
            self._x_dev[slot] = x               # keep alive until the forward has consumed it
        else:
            x = units
        t.fwd_events = None
        if self.time_forward:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(cur)
        # uint8 windows (b, L+1, H, W): pre-processing fused into the head conv (V2ce3d.forward_frames)
        with torch.cuda.stream(cur), nvtx('v2ce:unet'):
            if self.infer is not None:
                y = self.infer(x)
            else:
                y = self.model.forward_frames(x) if x.dtype == torch.uint8 else self.model(x)
        if self.time_forward:
            e1.record(cur)
            t.fwd_events = (e0, e1)
        b, L, _, H, W = y.shape
        n = b * L
        t.vox = y.reshape(n, 2, 10, H, W)
        if trim_last_window_to:                   # merge_voxels: drop the re-inferred overlap of the pulled-back window
            # a short image folder delivers a last window of fewer than `keep` pairs: the reference's [-mode:] slice
            # (v2ce.py:229-230) then keeps them all
            keep = min(trim_last_window_to, L)
            with torch.cuda.stream(cur):
                t.vox = torch.cat([t.vox[:(b - 1) * L], t.vox[(b - 1) * L + (L - keep):]], dim=0).contiguous()
            n = t.vox.shape[0]
        t.n_pairs, t.hw = n, (H, W)
        vox_ready = torch.cuda.Event()            # after the trim copy: the post stream reads t.vox
        vox_ready.record(cur)
        t.vox.record_stream(self.post_stream)
        self.launches += self.model.last_launches() if hasattr(self.model, 'last_launches') else 0

        # the batch before this one: its counts are on the host by the time UNet(i) is queued
        prev = self._pending
        if prev is not None:
            self._stage_b(prev)

        # stage A of this batch on the post stream, behind the network
        with torch.cuda.stream(self.post_stream), nvtx('v2ce:count+event-frame-sums'):
            self.post_stream.wait_event(vox_ready)
            eng = self.engines[slot]
            # keep_polarity: the per-polarity sums come out of the LDATI count pass below (one read of the voxels for
            # both stages); gray mode sums over both polarities and keeps its own pass
            fused = bool(self.keep)
            t.sums = torch.empty((n, 2, H, W), dtype=torch.float32, device=self.device) if fused else \
                _ef.accumulate(t.vox, self.keep)
            if keep_sums:
                self.sums.append(t.sums)
            small = self._buf(self._small_dev, slot, 8 * (4 + n * _ldati.NBINS)).view(torch.int64)
            t.params = _ldati.make_params(n, H, W, fps=self.fps, seed=self.seed, frame_base=pair_base,
                                          device=self.device, add_frame_offset=True)
            l0 = eng.launches
            seg = eng.count(t.vox, t.params, out=small[4:4 + n * _ldati.NBINS].view(n, _ldati.NBINS),
                            ef_sums=t.sums if fused else None)
            if self.per_batch_frames:
                nb = ctypes.c_size_t()
                check(self.lib.v2ce_ef_select_workspace_bytes(ctypes.byref(nb)))
                ws = self._buf(self._sel_ws, slot, nb.value)
                mult = 1 if self.keep else 3
                check(self.lib.v2ce_ef_select(ptr(t.sums), t.sums.numel(), float(self.percentile), mult, ptr(ws),
                                              ws.numel(), ptr(small), stream_ptr()))
            self.launches += (0 if fused else 1) + (4 if self.per_batch_frames else 0) + (eng.launches - l0)
            t.small_host = self._buf(self._small_host, slot, 8 * (4 + n * _ldati.NBINS), pinned=True).view(torch.int64)[
                :4 + n * _ldati.NBINS]
            t.small_host.copy_(small[:4 + n * _ldati.NBINS], non_blocking=True)
            offs_host = self._buf(self._offs_host, slot, 8 * n, pinned=True).view(torch.int64)[:n]
            offs_host.copy_(torch.from_numpy(_ldati.frame_offsets_us(pair_base, n, self.fps)))
            t.offs = self._buf(self._offs_dev, slot, 8 * n).view(torch.int64)[:n]
            t.offs.copy_(offs_host, non_blocking=True)
            t.counts_ready = torch.cuda.Event()
            t.counts_ready.record(self.post_stream)
        self._pending = t
        return t

    # ------------------------------------------------------------------------------------------
    def _stage_b(self, t):
        """Counts / order statistics of batch t are (about to be) on the host: size the outputs, enqueue
        normalise + emit/sort/pack on the post stream and the D2H of the results on the copy stream."""
        if t.staged:
            return
        t.counts_ready.synchronize()            # the one data-dependent sync: the counts size the output
        small = t.small_host.numpy()
        n, (H, W), slot = t.n_pairs, t.hw, t.slot
        t.seg_counts = small[4:].reshape(n, _ldati.NBINS).copy()
        total = int(t.seg_counts.sum())
        t.total = total
        t.ub = None
        frames = None
        with torch.cuda.stream(self.post_stream), nvtx('v2ce:emit+sort+pack'):
            if self.per_batch_frames:
                npos, lo, bits_lo, bits_hi = (int(v) for v in small[:4])
                if npos == 0:
                    raise ValueError('event frames hold no positive value: np.percentile of an empty array')
                mult = 1 if self.keep else 3
                a = np.array([bits_lo], dtype=np.uint32).view(np.float32)[0]
                b = np.array([bits_hi], dtype=np.uint32).view(np.float32)[0]
                t.ub = min(_ef.percentile_from_order_statistics(npos, mult, self.percentile, a, b), self.ceil)
                fr = self._buf(self._fr_dev, slot, n * H * W * 3)
                frames = _ef.normalize(t.sums, t.ub, self.keep, out=fr[:n * H * W * 3].view(n, H, W, 3))
                self.launches += 1
            eng = self.engines[slot]
            ev = self._buf(self._ev_dev, slot, max(total, 1) * 13)
            l0 = eng.launches
            # per-slot status words: a temporary would return to the post stream's pool while the copy stream
            # still has to read it
            st_dev = self._buf(self._st_dev, slot, 16).view(torch.int32)[:4]
            _, status = eng.emit(t.vox, t.params, total, frame_offsets=t.offs, out=ev, status_out=st_dev)
            self.launches += eng.launches - l0
            t.events_dev = ev
            t.frames_dev = frames
            t.packed = torch.cuda.Event()
            t.packed.record(self.post_stream)
        t.d2h_bytes = 0
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(t.packed)
            if self.collect_on_device and total > 0:
                need = self._all_bytes + total * 13
                self._pairs_collected += n
                if self._all_ev is None or self._all_ev.numel() < need:
                    # events per pair seen so far x the pairs of the whole clip (+15 %), at least double
                    est = int(need * max(self.clip_pairs, self._pairs_collected) / self._pairs_collected * 1.15)
                    grown = torch.empty(max(est if self.clip_pairs else 2 * need, need, 64 << 20), dtype=torch.uint8,
                                        device=self.device)
                    if self._all_bytes:
                        grown[:self._all_bytes].copy_(self._all_ev[:self._all_bytes])
                    self._all_ev = grown
                self._all_ev[self._all_bytes:need].copy_(ev[:total * 13])
                self._all_bytes = need
            t.ev_host = None
            if self.copy_out:
                if self.host_sink is not None:
                    evh = self.host_sink.place(slot, total * 13)
                else:
                    evh = self._buf(self._ev_host, slot, max(total, 1) * 13, pinned=True)
                evh[:total * 13].copy_(ev[:total * 13], non_blocking=True)
                t.ev_host = evh[:total * 13]
                t.d2h_bytes = total * 13 + (4 + n * _ldati.NBINS) * 8 + 16
                if frames is not None:
                    frh = self._buf(self._fr_host, slot, frames.numel(), pinned=True)
                    frh[:frames.numel()].copy_(frames.reshape(-1), non_blocking=True)
                    t.d2h_bytes += frames.numel()
            t.status = self._st_host[slot]
            t.status.copy_(status, non_blocking=True)   # pinned: a pageable target would block the host here
            t.done = torch.cuda.Event()
            t.done.record(self.copy_stream)
        self._free[slot] = t.done
        t.staged = True
        t.vox = None if not self.keep_vox else t.vox
        if self._pending is t:
            self._pending = None

    keep_vox = False                            # tests may set this to inspect the voxels a ticket was computed from

    def reset_collection(self, reserve_bytes=0):
        """Start a new clip: forget the events collected so far and any batch an aborted clip left half-way through
        the pipeline (its ticket would otherwise be staged into the new clip).  reserve_bytes > 0 sizes the device
        buffer up front (the caller's estimate from the schedule) so that it does not regrow by copy."""
        if self._pending is not None or any(f is not None for f in self._free):
            torch.cuda.synchronize(self.device)
        self._pending = None
        self._next = 0
        self._free = [None] * self.slots
        self.sums = []
        self._all_bytes = 0
        self._pairs_collected = 0
        if reserve_bytes and (self._all_ev is None or self._all_ev.numel() < reserve_bytes):
            self._all_ev = None
            self._all_ev = torch.empty(int(reserve_bytes), dtype=torch.uint8, device=self.device)

    def collected_events(self, to_host=True):
        """All events appended since reset_collection(), as (device uint8 tensor, host recarray view of one D2H or
        None when to_host is False)."""
        self.flush()
        self.copy_stream.synchronize()
        if self._all_bytes == 0:
            return None, (np.empty(0, _ldati.EVENT_DTYPE) if to_host else None)
        dev = self._all_ev[:self._all_bytes]
        from .sink import to_host as _sink
        return dev, (_sink(dev).view(_ldati.EVENT_DTYPE) if to_host else None)

    def flush(self):
        """Enqueue stage B of the batch submitted last (the end of a clip)."""
        if self._pending is not None:
            self._stage_b(self._pending)

    def wait(self, t, copy=True):
        """Block until batch `t` is on the host.  Returns (events recarray view, frames uint8 (n,H,W,3) | None);
        with copy_out=False both are None (results stay in the slot's device buffers, t.events_dev / t.frames_dev)."""
        self._stage_b(t)
        t.done.synchronize()
        _ldati.check_status(t.status.numpy())
        if not self.copy_out:
            return None, None
        ev = t.ev_host.numpy().view(_ldati.EVENT_DTYPE)
        fr = None
        if self.per_batch_frames:
            n, (H, W) = t.n_pairs, t.hw
            fr = self._fr_host[t.slot][:n * H * W * 3].numpy().reshape(n, H, W, 3)
        if copy:
            ev = ev.copy()
            fr = fr.copy() if fr is not None else None
        return ev, fr
