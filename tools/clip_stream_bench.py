"""ClipStream throughput and the window-assembly kernel on one GPU (profiles/clip_stream_bench.json).

    python tools/clip_stream_bench.py [--out result.json]      # prints the JSON result; --out also writes it

  stream    frame-pairs/s of the 321-frame 346 x 260 clip at -b 4 ('lively' synthetic checkpoint): ClipStream fed CUDA
            frames in pushes of 16, against stream_clip on the same frames in host memory (FakeVideoReader), alternating,
            each timed from the call to its last result on the host, with one warm-up run each
  assemble  v2ce_assemble_windows for one 64-pair batch (4 windows of 17 frames of 346 x 260, native route), gray and
            BGR: CUDA events around 200 launches that rotate over 8 batches of distinct frames (156 MB of BGR sources,
            more than the 126 MB L2); each call includes its pinned upload of the frame table, as ClipStream pays it;
            the HBM bound moves C*H*W bytes read plus H*W written per window frame at 7.7 TB/s

The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import synth  # noqa: E402
from oracle.ref_harness import FakeVideoReader  # noqa: E402

HBM_BPS = 7.7e12
N_FRAMES, H, W, L, B = 321, 260, 346, 16, 4


def _model():
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(31, 'lively'))
    return m.eval().to('cuda')


def run_stream_clip(model, frames):
    from v2ce_toolbox_b200 import v2ce as drv
    t0 = time.perf_counter()
    res = drv.stream_clip(model, vidcap=FakeVideoReader(frames), seq_len=L, width=W, height=H, batch_size=B, seed=0,
                          events_to_host=False)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res.n_pairs, res.n_events


def run_clip_stream(model, frames_dev):
    from v2ce_toolbox_b200 import ClipStream
    t0 = time.perf_counter()
    n_events = 0
    with ClipStream(model, seq_len=L, width=W, height=H, batch_size=B, seed=0) as cs:
        for a in range(0, len(frames_dev), 16):
            n_events += sum(b.n_events for b in cs.push(frames_dev[a:a + 16]))
        res = cs.close()
    n_events += sum(b.n_events for b in res.batches)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, res.n_pairs, n_events


def bench_assemble(color, reps=200):
    from v2ce_toolbox_b200 import frames as fr
    c = fr.COLORS[color][0]
    rng = np.random.default_rng(0)
    sets = []
    for _ in range(8):                                   # 8 batches of 65 distinct frames
        src = torch.from_numpy(rng.integers(0, 256, (65, H, W) + ((c,) if c > 1 else ()), dtype=np.uint8)).cuda()
        sets.append([src[i] for i in range(65)])
    slots = np.array([[k * L + j for j in range(L + 1)] for k in range(B)], np.int32)
    out = torch.empty((B, L + 1, H, W), dtype=torch.uint8, device='cuda')
    for s in sets:
        fr.assemble_windows(s, slots, color, 0, W, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fr.assemble_windows(sets[i % 8], slots, color, 0, W, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps                      # includes the per-call table upload
    window_frames = B * (L + 1)
    nbytes = window_frames * (c * H * W + H * W)
    return dict(color=color, ms_per_call=ms, bytes=nbytes, hbm_bound_ms=nbytes / HBM_BPS * 1e3,
                share_of_hbm_bound=nbytes / HBM_BPS * 1e3 / ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', help='also write the JSON result to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('clip_stream_bench: no CUDA device (nothing is measured without one)')
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    frames = synth.make_video(N_FRAMES, H, W, seed=1)
    frames_dev = torch.from_numpy(frames).cuda()
    m_a, m_b = _model(), _model()
    run_stream_clip(m_a, frames)                          # warm-up: modules, runner buffers, allocator
    run_clip_stream(m_b, frames_dev)
    rows = {'stream_clip_host_frames': [], 'clip_stream_device_frames': []}
    for _ in range(5):
        rows['stream_clip_host_frames'].append(run_stream_clip(m_a, frames))
        rows['clip_stream_device_frames'].append(run_clip_stream(m_b, frames_dev))
    result = {'gpu': q[0] if q else 'unknown', 'clip': dict(frames=N_FRAMES, height=H, width=W, seq_len=L, batch_size=B)}
    for k, v in rows.items():
        secs = [s for s, _, _ in v]
        result[k] = dict(seconds=secs, pairs=v[0][1], events=v[0][2], median_s=float(np.median(secs)),
                         pairs_per_s=v[0][1] / float(np.median(secs)))
    result['assemble'] = [bench_assemble('gray'), bench_assemble('bgr')]
    print(json.dumps(result, indent=1))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
