"""Batch windows from frames kept where the caller has them, with colour converted to gray on the device.

    assemble_windows(frames, slots, color, x0, out_width) -> (n_windows, L+1, H, out_width) uint8 CUDA

One launch of ``v2ce_assemble_windows`` (csrc/frames.cu).  ``frames`` is a list of uint8 CUDA tensors, (H, W) gray or
(H, W, C) colour; each may be a row- or column-cropped view with its own row pitch.  ``slots[w, j]`` is the index in
``frames`` of frame j of window w.  Colour becomes gray exactly as OpenCV's ``cvtColor(..., COLOR_*2GRAY)`` makes it
(oracle/frames_oracle.py).  The result is what ``V2ce3d.forward_frames`` (center crop, x0 = W // 2 - width // 2) and
``preprocess.image_units_device`` (full width) take.
"""
import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

# color name -> (channels, 1 when red comes first)
COLORS = {'gray': (1, 0), 'bgr': (3, 0), 'rgb': (3, 1), 'bgra': (4, 0), 'rgba': (4, 1)}


def frame_shape(color, height, width):
    """Shape of one frame of this colour order."""
    c = COLORS[color][0]
    return (height, width) if c == 1 else (height, width, c)


def device_frame(f, color):
    """`f` as the kernel reads it: the pixels of a row at a pitch of C bytes, the channels of a pixel adjacent.  A view
    with any other layout is copied into one that has it."""
    c = COLORS[color][0]
    if f.stride(-1) != 1 or (c > 1 and f.stride(-2) != c):
        f = f.contiguous()
    return f


def assemble_windows(frames, slots, color='gray', x0=0, out_width=None, out=None):
    c, rgb = COLORS[color]
    slots = np.ascontiguousarray(slots, dtype=np.int32)
    if slots.ndim != 2 or slots.size == 0 or slots.min() < 0 or slots.max() >= len(frames):
        raise _lib.V2ceError(f'slots must be a non-empty (n_windows, L+1) table of indices below {len(frames)}')
    shape = tuple(frames[0].shape)
    dev = frames[0].device
    if len(shape) != (2 if c == 1 else 3) or (c > 1 and shape[2] != c):
        raise _lib.V2ceError(f'{color} frames are {frame_shape(color, "H", "W")}, got {shape}')
    table = np.empty((len(frames), 2), np.int64)
    for i, f in enumerate(frames):
        _lib.require_cuda(f, 'frame')
        if f.dtype != torch.uint8 or tuple(f.shape) != shape or f.device != dev:
            raise _lib.V2ceError(f'frame {i}: expected uint8 {shape} on {dev}, got {f.dtype} {tuple(f.shape)} on {f.device}')
        if f.stride(-1) != 1 or (c > 1 and f.stride(-2) != c):
            raise _lib.V2ceError(f'frame {i}: strides {f.stride()} (pass it through device_frame)')
        table[i] = (f.data_ptr(), f.stride(0))
    H, W = shape[0], shape[1]
    out_width = W - x0 if out_width is None else out_width
    n, L1 = slots.shape
    with torch.cuda.device(dev):
        # one pinned upload of the frame table and the slots; the caching host allocator keeps the pinned copy alive
        # until the transfer has run
        host = torch.from_numpy(np.concatenate([table.reshape(-1), slots.reshape(-1).astype(np.int64)]))
        tab = host.pin_memory().to(dev, non_blocking=True)
        slots_dev = tab[2 * len(frames):].to(torch.int32)
        if out is None:
            out = torch.empty((n, L1, H, out_width), dtype=torch.uint8, device=dev)
        check(_lib.load().v2ce_assemble_windows(ptr(tab), ptr(slots_dev), n, L1, H, W, c, rgb, x0, out_width, ptr(out),
                                                stream_ptr()))
    return out
