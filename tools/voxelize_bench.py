"""events_to_voxels on one B200, against the torch path a user would otherwise write on the same card.

    python tools/voxelize_bench.py [--out result.json] [--reps 20]     # prints one JSON line; --out also writes it

Workloads (both 64 frames of 346 x 260 at fps 30, nbins 10: a 461 MB grid, larger than the 126 MB L2):
  clip      the device event stream of a 64-pair clip (stream_clip, events_to_host=False) of a synthetic 'lively'
            checkpoint on synth.make_video: frames in order, time-sorted within each LDATI bin segment;
  gt_like   a ground-truth-like stream with the same number of events in random order (uniform times, a moving blob,
            a 5 % hot pixel, polarities -1 / 0 / 1).
Each call writes the whole grid (memset) and reads every record once, so the HBM bound is (13 N + 4 F 2 nbins H W) bytes
over the data-sheet 7.7 TB/s of one HGX B200 GPU.  Timing: CUDA events around `reps` back-to-back calls after a warm-up;
the records (13 bytes per event: 2.1 GB for the clip's 160 M events) and the grid exceed L2, so no flush is needed.
The torch path decodes the columns, finds frames with torch.searchsorted, builds flat indices and runs torch.bincount,
then casts to float32; both paths must give identical tensors."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import synth_inputs as synth

H, W, PAIRS, FPS, NBINS = 260, 346, 64, 30, 10
HBM_BPS = 7.7e12                   # NVIDIA HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True, check=True).stdout.strip().split(', ')
    return {'name': q[0], 'power_limit': q[1]}


def clip_stream(device):
    from v2ce_toolbox_b200 import v2ce as drv
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(31, 'lively'))
    frames = synth.make_video(PAIRS + 1, H, W, seed=0)
    res = drv.stream_clip(m.eval().to(device), vidcap=synth.FakeVideoReader(frames), batch_size=4, fps=FPS, seed=0,
                          write_event_frames=False, events_to_host=False, device=device)
    return res.event_stream_dev


def gt_like_stream(n, edges, device):
    g = torch.Generator(device=device).manual_seed(7)
    e0, e1 = int(edges[0]), int(edges[-1])
    ts = torch.randint(e0, e1, (n,), generator=g, device=device, dtype=torch.int64)
    cx = (ts - e0).double() / (e1 - e0) * W
    x = (cx + torch.randn(n, generator=g, device=device, dtype=torch.float64) * (W / 20)).round().clamp(0, W - 1)
    y = (H / 2 + torch.randn(n, generator=g, device=device, dtype=torch.float64) * (H / 6)).round().clamp(0, H - 1)
    hot = torch.rand(n, generator=g, device=device) < 0.05
    x[hot], y[hot] = W // 3, H // 2
    p = torch.randint(-1, 2, (n,), generator=g, device=device, dtype=torch.int8)
    rec = torch.empty((n, 13), dtype=torch.uint8, device=device)
    rec[:, 0:8] = ts.view(torch.uint8).view(n, 8)
    rec[:, 8:10] = x.to(torch.int16).view(torch.uint8).view(n, 2)
    rec[:, 10:12] = y.to(torch.int16).view(torch.uint8).view(n, 2)
    rec[:, 12] = p.view(torch.uint8)
    return rec.reshape(-1)


def torch_voxels(rec, edges_dev, F, nbins, h, w):
    """The same convention in torch ops (events outside the sensor, with another polarity or outside the frames are
    dropped; the kernel also counts them)."""
    r = rec.view(-1, 13)
    ts = r[:, 0:8].contiguous().view(torch.int64).view(-1)
    x = r[:, 8:10].contiguous().view(torch.int16).view(-1).long()
    y = r[:, 10:12].contiguous().view(torch.int16).view(-1).long()
    p = r[:, 12].contiguous().view(torch.int8).long()
    keep = (x >= 0) & (x < w) & (y >= 0) & (y < h) & (p >= -1) & (p <= 1) & (ts >= edges_dev[0]) & (ts < edges_dev[-1])
    ts, x, y, p = ts[keep], x[keep], y[keep], p[keep]
    f = torch.searchsorted(edges_dev, ts, right=True) - 1
    e0 = edges_dev[f]
    c = ((ts - e0 + 1) * nbins - 1) // (edges_dev[f + 1] - e0)
    idx = (((f * 2 + (p != 1).long()) * nbins + c) * h + y) * w + x
    return torch.bincount(idx, minlength=F * 2 * nbins * h * w).float().view(F, 2, nbins, h, w)


def time_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    ap.add_argument('--reps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('voxelize_bench: no CUDA device (nothing is measured without one)')
    from v2ce_toolbox_b200 import _lib, events_to_voxels
    from v2ce_toolbox_b200.ldati import frame_offsets_us
    device = torch.device('cuda:0')
    torch.cuda.set_device(device)
    edges = frame_offsets_us(0, PAIRS + 1, FPS)              # the CLI's frame offsets, as events_to_voxels uses them
    edges_dev = torch.from_numpy(edges).to(device)
    cells = PAIRS * 2 * NBINS * H * W
    out = {'card': card(), 'hbm_bound_bandwidth': 'NVIDIA HGX B200 data sheet, 7.7 TB/s per GPU',
           'grid': [PAIRS, 2, NBINS, H, W], 'grid_bytes': 4 * cells, 'reps': args.reps, 'workloads': {}}
    clip = clip_stream(device)
    n = clip.numel() // 13
    lib = _lib.load()
    for name, rec in (('clip', clip), ('gt_like', gt_like_stream(n, edges, device))):
        ours = events_to_voxels(rec, PAIRS, FPS, nbins=NBINS)
        ref = torch_voxels(rec, edges_dev, PAIRS, NBINS, H, W)
        identical = bool(torch.equal(ours.view(torch.int32), ref.view(torch.int32)))
        assert identical, name
        del ours, ref
        vox = torch.empty((PAIRS, 2, NBINS, H, W), dtype=torch.float32, device=device)
        status = torch.empty(4, dtype=torch.int64, device=device)

        def kernel():
            _lib.check(lib.v2ce_events_to_voxels(_lib.ptr(rec), n, _lib.ptr(edges_dev), PAIRS, NBINS, H, W,
                                                 _lib.ptr(vox), _lib.ptr(status), _lib.stream_ptr()))
        row = {'events': n, 'identical_to_torch': identical}
        ms = time_ms(kernel, args.reps)
        torch_ms = time_ms(lambda: torch_voxels(rec, edges_dev, PAIRS, NBINS, H, W), max(args.reps // 4, 3), warm=1)
        byts = 13 * n + 4 * cells
        row.update({'ms': ms, 'gevents_per_s': n / ms / 1e6, 'bytes': byts, 'gb_per_s': byts / ms / 1e6,
                    'share_of_hbm_bound': byts / HBM_BPS / (ms / 1e3), 'torch_ms': torch_ms,
                    'speedup_over_torch': torch_ms / ms})
        out['workloads'][name] = row
        del vox
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
