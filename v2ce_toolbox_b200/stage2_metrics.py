"""Drop-in for the metric of /root/reference/train/scripts/stage2/stage2_metrics.py:22-88 on libv2ce_b200.so
(csrc/metrics.cu).

    ts_diff_metric(event_gt, event_pred, search_range=0, fps=30) -> np.array([mean distance in us, overflow count])

`event_gt` / `event_pred`: numpy record arrays with the fields timestamp, x, y, polarity (any integer widths; the packed
13-byte dtype of this toolbox is uploaded as it is) or uint8 CUDA tensors holding packed 13-byte records (what
``stream_clip(..., events_to_host=False)`` leaves on the device).  The sensor is 346 x 260 like the reference's
hard-coded lists; other sizes through ``width`` / ``height``.  The mean is (sum of exact integer distances + overflow *
cap) / n in float64: the reference adds the same terms one by one in Python floats, which can differ in the last bits."""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import V2ceError, check, ptr, stream_ptr
from .ldati import records_dev as _records_dev


def ts_diff_metric(event_gt, event_pred, search_range=0, fps=30, *, width=346, height=260, device=None):
    device = torch.device(device or 'cuda')
    if device.type != 'cuda':
        raise V2ceError('ts_diff_metric (B200) has no CPU path')
    lib = _lib.load()
    with torch.cuda.device(device):
        gt, n_gt = _records_dev(event_gt, device)
        pred, n_pred = _records_dev(event_pred, device)
        if n_gt == 0:
            raise ZeroDivisionError('ts_diff_metric: no ground-truth events')     # total_diff / gt_event_count upstream
        n = ctypes.c_size_t()
        check(lib.v2ce_ts_diff_workspace_bytes(width, height, n_pred, ctypes.byref(n)))
        ws = torch.empty(n.value, dtype=torch.uint8, device=device)
        res = torch.zeros(4, dtype=torch.int64, device=device)
        cap = 1e6 / fps / 10 * 3                                     # stage2_metrics.py:73
        check(lib.v2ce_ts_diff_metric(ptr(gt), n_gt, ptr(pred), n_pred, width, height, int(search_range), cap, ptr(ws),
                                      ws.numel(), ptr(res), stream_ptr()))
        total, overflow, bad_gt, bad_pred = (int(v) for v in res.cpu().tolist())
    if bad_gt or bad_pred:
        raise IndexError(f'ts_diff_metric: {bad_gt} ground-truth / {bad_pred} predicted events outside the {width}x{height} sensor')
    return np.array([(total + overflow * cap) / n_gt, overflow])
