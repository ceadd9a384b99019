#!/usr/bin/env python
"""bench.py -- V2CE hot path on B200: 346x260 frame-pairs/s (and LDATI Mevents/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): center 346x260, 321 synthetic gray frames = 20 windows of
16 frame pairs, batch 4, random-init V2ce3d, voxel + LDATI + event-frame path.  One *step* is one
batch of 4 windows (64 frame pairs) through v2ce_toolbox_b200.runner.BatchRunner: UNet ->
event-frame accumulate/select/normalise -> LDATI count/emit/sort/pack, the last two stages on a second
stream under the UNet of the next step.  Step i uses batch (i mod 5) of the clip; at N GPUs every rank
runs its own windows (weak scaling, windows are independent).

  value  device-timed throughput, inputs (float32 image units) already resident in HBM, results left on
         the device; at N > 1 the per-rank event shards are gathered to rank 0 over NCCL inside the timed
         region (dist.gather_event_shards: exact-length point-to-point transfers)
  e2e    same steps with HOST buffers: raw uint8 frame windows in pinned memory H2D (the pre-processing
         runs inside the head conv), packed events + preview frames D2H, inside the timed region; at N > 1
         every rank copies its own shard over its own PCIe link straight into its slice of a shared,
         page-locked host array that holds the merged stream (dist.SharedHostRing) -- no NCCL in this leg
  roofline    tensor roofline of the UNet forward (2169.336 GFLOP per window, SURVEY.md 8d): CUDA events around
              the forward run alone over the same K steps (`forward_ms`) and inside the timed steps
              (`forward_ms_in_step`); `frac` against the sustained bf16 peak, `frac_burst` against the burst peak
  ef          HBM roofline of the event-frame kernels (8,906,040 B per pair, SURVEY.md 8d)
  ldati       BASELINE configs[2]: LDATI alone on 1000 pairs of synthetic voxels (rand / randint10), in chunks,
              plus the 24- and 96-pair calls and the sparse distribution; HBM roofline
  library_baseline   the reference's own torch op sequence on the same GPU (torch_reference.py): cuDNN conv3d
              forward under TF32 and bf16 autocast, torch-CUDA LDATI, torch event frames
  clips       BASELINE configs[3]/[4]: the 9000-frame clip and the 600-frame 1920x1080 pano clip (2 tiles at the
              default height, 6 tiles at --height 1080) through dist.stream_clip_sharded at this N
  sharded_parity   (N > 1) sharded event stream + preview == single-process, bit for bit, checked before timing
  cpu_baseline     the CPU oracle (torch-CPU fp32 UNet + numpy LDATI/EF restatement, oracle/) timed on
              the host cores on a bounded sample (1 window = 16 frame pairs); N = 1 only

--dump-outputs DIR writes what the `value` path handed back in its last timed step (rank 0) as DIR/<name>.npy,
float32 / float64, under 40 MB: the per-(pair, bin) event counts, a fixed seeded sample of the event records, the
preview frames of a fixed seeded sample of the pairs and the preview's upper bound (dump_outputs).  Inputs, weights and
seeds are fixed, so two builds run with the same arguments can be compared file by file.

--impl reference times that CPU oracle port alone (the reference itself is Python and is not
present on the GPU box; oracle/ is pinned to it by tests/golden).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, L = 260, 346, 16
N_FRAMES = 321
BATCH = 4
GFLOP_PER_WINDOW = 2169.336
SHARD_CAP = 200 << 20                  # bytes reserved per rank and step for the merged event shards (150 MB expected)
EF_BYTES_PER_PAIR = 8_906_040          # SURVEY.md 8d: 80 B/pixel read + 8 sum write + 8 re-read + 3 uint8 write
METRIC = '346x260 frame-pairs/s (center, 321 frames, batch 4, voxel+LDATI+event-frame)'
# dram__bytes_read.sum + dram__bytes_write.sum of one V2ce3d forward (batch 4), summed over its launches from the
# ncu capture summarised in profiles/forward_traffic_r2.txt (tools/ncu_traffic.py)
TRAFFIC_BYTES = 13.24e9        # read 9.17 GB + write 4.06 GB (L2: 59.2 GB): profiles/forward_traffic_r2.txt
KERNEL_NOTE = ('V2ce3d forward (26 launches + 4 spectral-norm launches on a side stream): conv_halo_kdm_kernel x11 '
               '(head, stride-2 encoder convs and decoder convs with fused shortcuts, N<=64 convs), conv_halo_kernel x10, '
               'conv_igemm_kernel x4 (remaining 1x1x1 shortcuts, side stream), head prep')


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {'tf': d.get('bf16_tflops_sustained', 1390.9), 'tf_burst': d.get('bf16_tflops', 1657.0),
                'hbm': d.get('hbm_gbs', 6531.6), 'source': 'measured'}
    return {'tf': 1400.0, 'tf_burst': 1650.0, 'hbm': 6650.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {'sm_mhz': float(np.median(busy)) if busy else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def make_inputs():
    """The 20 windows of the clip: preprocessed image units (20, 16, 2, 260, 346) float32 and the raw gray frames
    they come from (20, 17, 260, 346) uint8 (both host)."""
    import synth_inputs as synth
    from v2ce_toolbox_b200.v2ce import image_pre_processing, window_schedule
    frames = synth.make_video(N_FRAMES, H, W, seed=0)
    starts, mode = window_schedule(N_FRAMES, L)
    assert mode == 0 and len(starts) == 20
    units = torch.stack([image_pre_processing(frames[s:s + L + 1], H) for s in starts], dim=0)
    windows = torch.from_numpy(np.stack([frames[s:s + L + 1] for s in starts], axis=0))     # (20, 17, H, W) uint8
    return units, windows


# ------------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------------
def cpu_port_step(orc, units_window, pair_base, fps=30):
    from oracle import ef_oracle, ldati_oracle
    vox = orc.forward(units_window).numpy().reshape(-1, 2, 10, H, W)
    frames, _, _ = ef_oracle.event_frames_oracle(vox, 10, 98, True)
    ev = ldati_oracle.sample_voxel_statistical_oracle(vox, fps=fps, seed=0, frame_base=pair_base, flavor='cpu')
    return sum(len(e) for e in ev)


def time_cpu_port(units, steps, warmup):
    import synth_inputs as synth
    from oracle.unet_oracle import UNetOracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    orc = UNetOracle(synth.make_state_dict(0, 'reference'))
    for i in range(warmup):
        cpu_port_step(orc, units[i % 20:i % 20 + 1], 0)
    t0 = time.perf_counter()
    events = 0
    for i in range(steps):
        events += cpu_port_step(orc, units[i % 20:i % 20 + 1], (i % 20) * L)
    dt = time.perf_counter() - t0
    return steps * L / dt, events / dt / 1e6, dt, cores


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    units, _ = make_inputs()
    # one window (16 pairs) per step: a step takes seconds on the host cores
    steps, warmup = args.steps, args.warmup
    pairs_s, mev_s, dt, cores = time_cpu_port(units, steps, warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': pairs_s, 'unit': 'frame-pairs/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warmup, 'ms_per_step': dt / steps * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'center 346x260, 321 frames, batch 4, voxel+LDATI+event-frame video',
                   'sample': '1 window (16 frame pairs) per step on host cores'},
        'cpu_baseline': {'value': pairs_s, 'unit': 'frame-pairs/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{steps} steps x 1 window (16 pairs): torch-CPU fp32 UNet + numpy LDATI/EF oracle'},
        'e2e': {'value': pairs_s, 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'ldati_mevents_per_s': mev_s, 'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def new_model(device, seed=0, init='reference'):
    import synth_inputs as synth
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(seed, init))
    return m.eval().to(device)


class Runner:
    """Model + two BatchRunners (v2ce_toolbox_b200.runner): device-resident inputs / results for `value`,
    pinned host inputs and host results for `e2e`."""

    def __init__(self, device, units_host, windows_host, rank, world):
        from v2ce_toolbox_b200.runner import BatchRunner
        self.device = device
        self.rank, self.world = rank, world
        self.model = new_model(device)
        self.dev_runner = BatchRunner(self.model, device, fps=30, seed=0, copy_out=False)
        self.host_runner = BatchRunner(self.model, device, fps=30, seed=0, copy_out=True)
        self.dev_runner.time_forward = True
        # value: image units resident in HBM; e2e: the raw uint8 windows in pinned host memory (the pre-processing
        # of v2ce.py:45-64 runs inside the head conv, V2ce3d.forward_frames)
        self.units_dev = [units_host[i:i + BATCH].contiguous().to(device) for i in range(0, 20, BATCH)]
        self.units_pinned = [windows_host[i:i + BATCH].contiguous().pin_memory() for i in range(0, 20, BATCH)]
        self.n_pairs = BATCH * L
        self.comm_stream = torch.cuda.Stream(device=device) if world > 1 else None
        self.gather_bufs = [None, None]           # rank 0: merged shards of alternate steps
        self.gathers = 0
        self.ring_note = None
        self.window, self.gather_note = None, None
        if world > 1:
            from v2ce_toolbox_b200 import dist as vdist
            if os.environ.get('V2CE_BENCH_GATHER', 'p2p') == 'p2p':
                try:
                    # merged shards of alternate steps live in two buffers on rank 0 that every rank maps (CUDA IPC)
                    self.window = vdist.PeerWindow(world * SHARD_CAP, buffers=2, device=device)
                    self.gather_note = 'copy-engine pushes into a peer window on rank 0 (dist.PeerWindow, CUDA IPC over NVLink)'
                except Exception as e:                 # noqa: BLE001 -- raised on every rank alike
                    self.gather_note = f'NCCL point-to-point gather (dist.gather_event_shards; no peer window: {e})'
            else:
                self.gather_note = 'NCCL point-to-point gather to rank 0 (dist.gather_event_shards)'
            try:
                # merged events of one step: ~180 k events per pair x 64 pairs x 13 B = 150 MB per rank; one slot
                # per runner slot
                self.host_runner.host_sink = vdist.SharedHostRing(self.host_runner.slots, world * SHARD_CAP)
                self.ring_note = 'shared page-locked host ring (dist.SharedHostRing)'
            except Exception as e:                     # noqa: BLE001 -- e2e then uses per-rank pinned buffers
                self.ring_note = f'per-rank pinned buffers ({type(e).__name__}: {e})'

    def gather(self, t):
        """Final gather of the per-rank event shards of batch t to rank 0 (NCCL over NVLink, the product's
        dist.gather_event_shards) on the comm stream, behind the pack kernel."""
        from v2ce_toolbox_b200 import dist as vdist
        k = self.gathers & 1
        self.gathers += 1
        if self.window is not None:
            # counts over the host group, then ONE asynchronous copy per rank on the comm stream: no kernel at all.
            # The merged buffer is complete on rank 0 once every rank's stream has drained (the barrier that closes
            # the timed region; dist.gather_event_shards(window=...) is the blocking form).
            counts = vdist.exchange_counts(t.total)
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(t.packed)
                self.window.push(k, t.events_dev, counts, vdist.EVENT_BYTES)
                fin = torch.cuda.Event()
                fin.record(self.comm_stream)
            return fin
        with torch.cuda.stream(self.comm_stream):
            # its own stream: the post stream already holds stage A of the next batch, which waits for the next UNet.
            # Nothing here waits on the device: the counts travel over the host-side gloo group, the shards as
            # asynchronous point-to-point transfers that run when an SM has room for NCCL's CTAs.
            self.comm_stream.wait_event(t.packed)
            if self.rank == 0 and self.gather_bufs[k] is None:
                self.gather_bufs[k] = torch.empty(self.world * SHARD_CAP, dtype=torch.uint8, device=self.device)
            merged, counts = vdist.gather_event_shards(t.events_dev, t.total, out=self.gather_bufs[k])
            fin = torch.cuda.Event()
            fin.record(self.comm_stream)
        return fin


def check_sharded_parity(device, rank, world):
    """Before any timing at N > 1: the sharded path (windows / pano windows over ranks, spectral-norm replay, shard
    merge in host shared memory and over NCCL, preview from gathered sums) equals the single-process path bit for bit.
    The driver's GPU test box has one GPU and skips tests/test_gpu_dist.py, so the same check runs here."""
    import torch.distributed as dist
    import synth_inputs as synth
    from v2ce_toolbox_b200 import dist as vdist, v2ce as drv
    cases = {'center': (16 * 2 * world + 9, 28, 36, 'center', 36, 28, 1),
             'center_b2': (16 * 4 * world + 1, 28, 36, 'center', 36, 28, 2),
             'pano': (16 * (world + 1) + 8, 24, 80, 'pano', 32, 24, 1),
             # one window, fewer batches than ranks: its three width tiles are shared among the ranks (dist.pano_tile_owner)
             'pano_tiles': (17, 24, 80, 'pano', 32, 24, 1)}
    out = {}
    for name, (n_frames, h, w, infer_type, width, height, bs) in cases.items():
        frames = synth.make_video(n_frames, h, w, seed=5)
        kw = dict(seq_len=16, batch_size=bs, infer_type=infer_type, width=width, height=height, fps=30, seed=9)
        preview = {}
        ev, n = vdist.stream_clip_sharded(new_model(device, 31, 'lively'), synth.FakeVideoReader(frames), n_frames, world,
                                          rank, device=device, preview=preview, ceil=10, upper_bound_percentile=98, **kw)
        ev_dev, n2 = vdist.stream_clip_sharded(new_model(device, 31, 'lively'), synth.FakeVideoReader(frames), n_frames,
                                               world, rank, device=device, to_host=False, **kw)
        ok = torch.ones(1, dtype=torch.int64, device=device)
        if rank == 0:
            res = drv.stream_clip(new_model(device, 31, 'lively'), vidcap=synth.FakeVideoReader(frames), device=device,
                                  write_event_frames=True, ceil=10, upper_bound_percentile=98, **kw)
            want = res.event_stream.view(np.uint8)
            same = (n == n2 == len(res.event_stream) > 0 and np.array_equal(np.asarray(ev).view(np.uint8), want) and
                    np.array_equal(ev_dev.cpu().numpy(), want) and
                    preview['upper_bound'] == res.ef_upper_bound and np.array_equal(preview['frames'], res.ef_frames))
            ok[0] = 1 if same else 0
            out[name] = {'events': int(n), 'pairs': n_frames - 1, 'equal': bool(same)}
        dist.broadcast(ok, src=0)
        if int(ok.item()) != 1:
            raise AssertionError(f'sharded_parity: {name} differs from the single-process stream at {world} ranks')
    # the per-step merge `value` times: copy-engine pushes into a peer window == the NCCL point-to-point gather
    try:
        win = vdist.PeerWindow(1 << 20, buffers=1, device=device)
    except Exception as e:                             # noqa: BLE001 -- raised on every rank alike
        out['peer_window'] = {'available': False, 'why': str(e)[:200]}
        return out
    ok = torch.ones(1, dtype=torch.int64, device=device)
    for step, n in enumerate([3000 + 11 * rank, 0 if rank == 0 else 7, 0]):
        g = torch.Generator().manual_seed(1000 * step + rank)
        shard = torch.randint(0, 256, (n * 13 + 16,), dtype=torch.uint8, generator=g).to(device)
        a, _ = vdist.gather_event_shards(shard, n)
        b, counts = vdist.gather_event_shards(shard, n, window=win)
        if rank == 0 and not (b.numel() == sum(counts) * 13 and torch.equal(a, b)):
            ok[0] = 0
    win.close()
    dist.broadcast(ok, src=0)
    if int(ok.item()) != 1:
        raise AssertionError(f'sharded_parity: peer-window merge differs from the NCCL gather at {world} ranks')
    out['peer_window'] = {'available': True, 'equal': True}
    return out


DUMP_EVENTS = 1 << 20                  # event records sampled by --dump-outputs
DUMP_PAIRS = 8                         # frame pairs whose preview frames --dump-outputs keeps


def dump_outputs(out_dir, t):
    """The results of BatchRunner ticket t as out_dir/<name>.npy: the event counts per (pair, bin), DUMP_EVENTS event
    records at seeded sorted positions of the packed stream (all of them when there are fewer), the preview frames of
    DUMP_PAIRS seeded pairs and the preview's upper bound.  Under 40 MB whatever the event count."""
    from v2ce_toolbox_b200.ldati import EVENT_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    n = t.seg_counts.shape[0]
    pairs = np.sort(rng.choice(n, min(n, DUMP_PAIRS), replace=False))
    rows = np.arange(t.total) if t.total <= DUMP_EVENTS else np.sort(rng.choice(t.total, DUMP_EVENTS, replace=False))
    packed = t.events_dev[:t.total * EVENT_DTYPE.itemsize].view(t.total, EVENT_DTYPE.itemsize)
    ev = packed.index_select(0, torch.from_numpy(rows).to(packed.device)).cpu().numpy().reshape(-1).view(EVENT_DTYPE)
    frames = t.frames_dev[torch.from_numpy(pairs).to(t.frames_dev.device)].cpu().numpy()
    out = {'events_per_pair_bin': t.seg_counts.astype(np.float64), 'events_index': rows.astype(np.float64),
           'events_timestamp': ev['timestamp'].astype(np.float64), 'events_x': ev['x'].astype(np.float32),
           'events_y': ev['y'].astype(np.float32), 'events_polarity': ev['polarity'].astype(np.float32),
           'event_frames_pairs': pairs.astype(np.float64), 'event_frames': frames.astype(np.float32),
           'event_frames_upper_bound': np.array([t.ub], np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    device = torch.device('cuda', local_rank)
    torch.cuda.set_device(device)
    affinity = None
    if world > 1:
        # one process per GPU: keep each rank (and the pinned staging it allocates) on its GPU's NUMA node
        from v2ce_toolbox_b200.dist import bind_to_gpu_numa
        affinity = bind_to_gpu_numa(local_rank)
    parity = None
    if world > 1:
        parity = check_sharded_parity(device, rank, world)
    units, windows = make_inputs()
    r = Runner(device, units, windows, rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(host_io):
        """One step = one batch of 4 windows through BatchRunner.submit; the results of step i are collected
        (and, at N > 1, merged: NCCL gather to rank 0 for `value`, shared host array for `e2e`) while step i+1
        computes."""
        br = r.host_runner if host_io else r.dev_runner
        src = r.units_pinned if host_io else r.units_dev
        stats = {'events': 0, 'fwd': [], 'gap': [], 'h2d': 0, 'd2h': 0, 'last_fwd_end': None, 'last': None}
        pending = []                               # gathers in flight (their buffers alternate: wait for the one before last)

        def collect(t, timed):
            br.wait(t, copy=False)
            if world > 1 and not host_io:
                pending.append(r.gather(t))
                if len(pending) > 1:
                    pending.pop(0).synchronize()
            if timed:
                stats['events'] += t.total
                stats['h2d'], stats['d2h'] = t.h2d_bytes, t.d2h_bytes
                if t.fwd_events is not None:
                    stats['fwd'].append(t.fwd_events[0].elapsed_time(t.fwd_events[1]))
                    if stats['last_fwd_end'] is not None:       # main-stream time between two networks
                        stats['gap'].append(stats['last_fwd_end'].elapsed_time(t.fwd_events[0]))
                    stats['last_fwd_end'] = t.fwd_events[1]

        def run(n, timed):
            prev = None
            for i in range(n):
                b = i % 5
                t = br.submit(src[b], (rank * 5 + b) * r.n_pairs)
                if prev is not None:
                    collect(prev, timed)
                prev = t
            if prev is not None:
                collect(prev, timed)
                stats['last'] = prev
            while pending:
                pending.pop(0).synchronize()

        run(args.warmup, False)
        br.launches = 0
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record()
        run(args.steps, True)
        torch.cuda.synchronize()
        e.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max(s.elapsed_time(e), wall * 1e3) if host_io else s.elapsed_time(e)
        tt = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()), stats, br.launches

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, st_dev, launches = timed_loop(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st_dev['last'])
    ms_e2e, st_e2e, _ = timed_loop(True)
    # the network alone (no event-frame / LDATI kernels sharing the SMs): what the roofline fraction describes
    fwd_ms = []
    for i in range(3):                          # untimed: the timed steps ran the network on the runner's own stream, so
        r.model(r.units_dev[i % 5])             # this stream's allocator pool has no 460 MB output block yet
    torch.cuda.synchronize()
    for i in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r.model(r.units_dev[i % 5])
        e1.record()
        fwd_ms.append((e0, e1))
    torch.cuda.synchronize()
    fwd_alone = float(np.mean([a.elapsed_time(b) for a, b in fwd_ms]))
    clocks = sampler.stop() if rank == 0 else None
    link = host_link_probe(device) if rank == 0 else None

    pairs_per_step = r.n_pairs * world
    value = pairs_per_step * args.steps / (ms_dev / 1e3)
    e2e = pairs_per_step * args.steps / (ms_e2e / 1e3)
    pk = peaks()
    fwd_in_step = float(np.mean(st_dev['fwd'])) if st_dev['fwd'] else float('nan')
    fwd = fwd_alone
    achieved = GFLOP_PER_WINDOW * BATCH / fwd            # GFLOP / ms = TFLOP/s
    line = {
        'metric': METRIC, 'value': value, 'unit': 'frame-pairs/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': 'center 346x260, 321 frames, batch 4, voxel+LDATI+event-frame video',
                   'pairs_per_step_per_gpu': r.n_pairs, 'weights': 'random-init V2ce3d (seed 0)',
                   'l2': 'inputs+activations per step (2.6 GB) exceed the 126 MB L2',
                   'pipeline': 'event frames + LDATI of step i run on a second stream under the UNet of step i+1',
                   'e2e_input': 'uint8 gray frame windows (4 x 17 x 260 x 346) in pinned host memory; pre-processing '
                                'fused into the head conv; events + preview frames copied back to pinned host memory',
                   'multi_gpu': 'windows sharded per rank; value: ' + (r.gather_note or 'n/a') + '; e2e: ' +
                                (r.ring_note or 'n/a')},
        'e2e': {'value': e2e, 'unit': 'frame-pairs/s', 'h2d_bytes_per_step': st_e2e['h2d'],
                'd2h_bytes_per_step': st_e2e['d2h'], 'ms_per_step': ms_e2e / args.steps, 'host_link': link},
        'gpu_launches': launches,
        'ldati_mevents_per_s': st_dev['events'] * world / (ms_dev / 1e3) / 1e6,
        'events_per_pair': st_dev['events'] / (r.n_pairs * args.steps),
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': pk['tf'], 'unit': 'TFLOP/s',
                     'frac': achieved / pk['tf'], 'peak_burst': pk['tf_burst'], 'frac_burst': achieved / pk['tf_burst'],
                     'traffic': TRAFFIC_BYTES, 'peak_source': pk['source'], 'kernel': KERNEL_NOTE,
                     'forward_ms': fwd, 'forward_ms_in_step': fwd_in_step,
                     'frac_in_step': GFLOP_PER_WINDOW * BATCH / fwd_in_step / pk['tf'],
                     'forward_share_of_step': fwd / (ms_dev / args.steps),
                     'forward_gap_ms_in_step': float(np.mean(st_dev['gap'])) if st_dev['gap'] else None,
                     'note': 'forward_ms: CUDA events around the network run alone over the same K steps; '
                             'forward_ms_in_step: the same events inside the timed steps, where the previous '
                             'batch\'s event-frame / LDATI kernels share the SMs.  peak = sustained cuBLAS bf16 '
                             '(clocks under a long run), peak_burst = its best-of-10 figure: a short run like this '
                             'one holds burst clocks, so frac_burst is the conservative fraction'},
        'cpu_baseline': None,
        'clocks': clocks,
        'cpu_affinity': None if affinity is None else {'cpus': len(affinity), 'first': affinity[0], 'last': affinity[-1]},
    }
    if parity is not None:
        line['sharded_parity'] = True
        line['sharded_parity_cases'] = parity
    if r.host_runner.host_sink is not None:
        r.host_runner.host_sink.close()
    if r.window is not None:
        r.window.close()
    del r.dev_runner, r.host_runner
    free_device_memory()

    def guarded(key, fn, timeout_s=600):
        """Secondary records must never cost the headline line: an exception becomes an `error` entry, and a record
        that does not return within `timeout_s` (a collective some rank never reached) makes every rank's own watchdog
        print what there is (rank 0) and leave."""
        def bail():
            line[key] = {'error': f'no result within {timeout_s} s; process ended by the watchdog'}
            if rank == 0:
                print(json.dumps(line), flush=True)
            os._exit(0)
        dog = threading.Timer(timeout_s, bail)
        dog.daemon = True
        dog.start()
        try:
            line[key] = fn()
        except Exception as e:                      # noqa: BLE001
            line[key] = {'error': f'{type(e).__name__}: {e}'}
        finally:
            dog.cancel()
        free_device_memory()

    if not args.headline_only:
        if world == 1:
            guarded('ef', lambda: ef_record(device, pk['hbm']))
            guarded('ldati', lambda: ldati_microbench(device, pk['hbm']))
            guarded('library_baseline', lambda: library_baseline(device, r.units_dev, fwd, line.get('ldati'), line.get('ef')))
        # every rank takes part (collectives inside); only rank 0 keeps the record
        guarded('clips', lambda: clips_record(device, rank, world, args), timeout_s=420)
        if world == 1 and not args.no_cpu_baseline:
            def cpu():
                pairs_s, mev_s, dt, cores = time_cpu_port(units, 2, 1)
                return {'value': pairs_s, 'unit': 'frame-pairs/s', 'cores': cores, 'kind': 'port',
                        'sample': '2 steps x 1 window (16 pairs): torch-CPU fp32 UNet + numpy LDATI/EF oracle',
                        'ldati_mevents_per_s': mev_s,
                        'extrapolated_s': {'long clip (8999 pairs)': 8999 / pairs_s,
                                           'pano 2 tiles (599 pairs x 2 model calls)': 599 * 2 / pairs_s,
                                           'note': 'SURVEY.md 8d config 5: the reference cannot hold a 9000-frame clip '
                                                   '(>130 GB of host voxels); extrapolated from the sample at its '
                                                   'pairs/s, pano counted per 346-px tile call'}}
            guarded('cpu_baseline', cpu)
    if rank == 0:
        print(json.dumps(line), flush=True)


def host_link_probe(device, mb=160, reps=5):
    """Pinned D2H / H2D rate of this box with the GPU otherwise idle (160 MB = one step's results).  The e2e leg hides a
    step's D2H behind the next step's network only while that copy is shorter than the network (9 ms: 18 GB/s); on a
    box whose host side delivers less (shared PCIe switch / host memory: 11-12 GB/s measured on some) e2e is the
    copy, not the GPU -- this record says which case the line was measured in."""
    dev = torch.empty(mb << 20, dtype=torch.uint8, device=device)
    host = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)
    out = {'mb': mb}
    for key, (dst, src) in (('d2h_gbs', (host, dev)), ('h2d_gbs', (dev, host))):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        out[key] = (mb << 20) * reps / (e0.elapsed_time(e1) / 1e3) / 1e9
    return out


def free_device_memory():
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def _time_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def ef_record(device, hbm_peak, n=64, reps=10):
    """Event frames alone on one batch of 64 frame pairs of voxels: accumulate -> exact percentile select -> normalise.
    Algorithmic bytes (SURVEY.md 8d): 8,906,040 per pair."""
    from v2ce_toolbox_b200 import event_frames as ef
    g = torch.Generator(device=device).manual_seed(1)
    vox = torch.rand((n, 2, 10, H, W), generator=g, device=device) * 0.02
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def run():
        flush.zero_()                              # voxels (461 MB) exceed the 126 MB L2 anyway; this evicts the sums
        return ef.event_frames(vox, 10, 98, True)

    ms_all = _time_ms(run, reps)
    ms_flush = _time_ms(lambda: flush.zero_(), reps)
    ms = ms_all - ms_flush
    alg = n * EF_BYTES_PER_PAIR
    return {'bound': 'hbm', 'pairs': n, 'ms': ms, 'achieved': alg / ms / 1e6, 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': alg / ms / 1e6 / hbm_peak, 'algorithmic_bytes': alg, 'pairs_per_s': n / ms * 1e3,
            'includes': 'the host read of the order statistics between select and normalise (one sync)'}


def ldati_microbench(device, hbm_peak, reps=5):
    """BASELINE.json configs[2]: LDATI alone on synthetic event-count voxels 346x260x10 bins, distributions (a) torch.rand
    and (b) randint(0,10) taken from the reference's own bench (LDATI.py:327-346) and (c) 0.015*rand (sparse, the regime
    of a random-init network).  `*_1000pairs`: the full 1000 pairs, resident on the device (7.2 GB), processed in chunks
    of 100 pairs (the reference chunks by 24, v2ce.py:301 -- its dense (B,2,9,H,W,M) tensors do not fit more; this path
    holds one 4-byte word per event).  Also single calls of 24 and 96 pairs.  Device-timed count -> (counts D2H) ->
    emit/sort/pack; HBM roofline with SURVEY.md 8d's algorithmic bytes: 4*20*H*W per pair read + 13 B per event written."""
    from v2ce_toolbox_b200 import ldati
    eng = ldati.LdatiEngine(device)
    out = {}

    def gen(name, F, seed=42):
        g = torch.Generator(device=device).manual_seed(seed)
        if name == 'rand':
            return torch.rand((F, 2, 10, H, W), generator=g, device=device)
        if name == 'sparse':
            return torch.rand((F, 2, 10, H, W), generator=g, device=device) * 0.015
        return torch.randint(0, 10, (F, 2, 10, H, W), generator=g, device=device).float()

    def record(F, total, ms):
        alg = F * 4 * 20 * H * W + 13 * total
        return {'pairs': F, 'events_per_pair': total / F, 'ms': ms, 'mevents_per_s': total / ms / 1e3,
                'pairs_per_s': F / ms * 1e3, 'algorithmic_bytes': alg, 'achieved_gbs': alg / ms / 1e6,
                'frac_of_hbm_peak': alg / ms / 1e6 / hbm_peak}

    for F in (24, 96):
        for name in ('rand', 'randint10') + (('sparse',) if F == 24 else ()):
            vox = gen(name, F)
            params = ldati.make_params(F, H, W, fps=30, seed=42, frame_base=0, device=device)
            total = [0]

            def run():
                _, seg, _ = eng.run(vox, params)
                total[0] = int(seg.sum())
            ms = _time_ms(run, reps)
            out[name if F == 24 else f'{name}_{F}pairs'] = record(F, total[0], ms)
            del vox
    chunk = 100
    for name in ('rand', 'randint10'):
        vox = torch.empty((1000, 2, 10, H, W), dtype=torch.float32, device=device)
        for i in range(0, 1000, chunk):
            vox[i:i + chunk] = gen(name, chunk, seed=42 + i)
        plist = [ldati.make_params(chunk, H, W, fps=30, seed=42, frame_base=i, device=device) for i in range(0, 1000, chunk)]
        total = [0]

        def run_all():
            total[0] = 0
            for k, i in enumerate(range(0, 1000, chunk)):
                _, seg, _ = eng.run(vox[i:i + chunk], plist[k])
                total[0] += int(seg.sum())
        ms = _time_ms(run_all, 2, warm=1)
        out[f'{name}_1000pairs'] = {**record(1000, total[0], ms), 'chunk_pairs': chunk}
        del vox
    return out


def library_baseline(device, units_dev, ours_forward_ms, ldati_rec, ef_rec):
    """SURVEY.md 8d / 2c: the reference's own torch op sequence on this GPU (torch_reference.py -- /root/reference is
    Python calling torch; it is not on this box, so its calls are re-issued one for one): cuDNN conv3d forward in
    upstream's default mode (TF32 allowed) and under bf16 autocast, torch-CUDA LDATI on the reference's 24-pair chunk,
    and the event-frame arithmetic with torch ops.  Kernel to beat = cuDNN / ATen / cub."""
    import synth_inputs as synth
    import torch_reference as tr
    out = {'torch': torch.__version__, 'cudnn': torch.backends.cudnn.version()}
    sd = synth.make_state_dict(0, 'reference')
    x = units_dev[0]
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        torch.backends.cudnn.benchmark = True
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cuda.matmul.allow_tf32 = True
        ref = tr.TorchV2ce3d(sd, device)
        ms_tf32 = _time_ms(lambda: ref(x), 5, warm=3)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            ms_bf16 = _time_ms(lambda: ref(x), 5, warm=3)
        del ref
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    out['unet_forward_batch4'] = {
        'cudnn_tf32_ms': ms_tf32, 'cudnn_bf16_autocast_ms': ms_bf16, 'ours_ms': ours_forward_ms,
        'cudnn_tf32_tflops': GFLOP_PER_WINDOW * BATCH / ms_tf32, 'cudnn_bf16_tflops': GFLOP_PER_WINDOW * BATCH / ms_bf16,
        'ours_over_cudnn_tf32': ms_tf32 / ours_forward_ms, 'ours_over_cudnn_bf16': ms_bf16 / ours_forward_ms,
        'note': 'same random-init weights and input batch (4 x 16 x 2 x 260 x 346); conv3d + batch_norm + relu as separate '
                'launches like the reference modules, cudnn.benchmark on; NCDHW fp32 tensors as the reference holds them'}
    free_device_memory()
    for name in ('rand', 'randint10'):
        g = torch.Generator(device=device).manual_seed(42)
        vox = torch.rand((24, 2, 10, H, W), generator=g, device=device) if name == 'rand' else \
            torch.randint(0, 10, (24, 2, 10, H, W), generator=g, device=device).float()
        n_ev = [0]

        def run():
            res = tr.sample_voxel_statistical_torch(vox, fps=30, stable=False, to_numpy=False)
            n_ev[0] = sum(int(r[0].shape[0]) for r in res)
        t0 = time.perf_counter()
        ms = _time_ms(run, 2, warm=1)
        ours = (ldati_rec or {}).get(name, {}).get('ms')
        out[f'ldati_{name}_24pairs'] = {'torch_cuda_ms': ms, 'events': n_ev[0], 'torch_cuda_mevents_per_s': n_ev[0] / ms / 1e3,
                                        'ours_ms': ours, 'ours_over_torch_cuda': (ms / ours) if ours else None,
                                        'note': 'events left on the device on both sides (the reference also copies four '
                                                'columns per frame to the host, LDATI.py:305)'}
        del vox
        free_device_memory()
    g = torch.Generator(device=device).manual_seed(1)
    vox = torch.rand((64, 2, 10, H, W), generator=g, device=device) * 0.02
    ms = _time_ms(lambda: tr.event_frames_torch(vox, 10, 98, True), 3, warm=1)
    ours = (ef_rec or {}).get('ms')
    out['event_frames_64pairs'] = {'torch_cuda_ms': ms, 'ours_ms': ours, 'ours_over_torch_cuda': (ms / ours) if ours else None,
                                   'note': 'the reference does this step in numpy on the host (v2ce.py:241-280); '
                                           'torch.quantile on a 16 M-element prefix (its input limit)'}
    return out


def clips_record(device, rank, world, args):
    """BASELINE configs[4] (long clip: center 346x260, 9000 frames, temporal windows sharded over the ranks, event merge)
    and configs[3] (pano 1920x1080, 600 frames: variant A = default --height 260 -> 462x260 -> 2 tiles; variant B =
    --height 1080 -> 6 tiles of 346x1080) through dist.stream_clip_sharded.  Per clip: `device` = all ranks computed and
    the shards merged on rank 0's GPU over NCCL (to_host=False); `e2e` = the merged stream in ONE host array, copied down
    from rank 0's GPU after the NCCL merge; `e2e_shm_merge` (N > 1) = the same array in POSIX shared memory, every rank
    copying its shard over its own PCIe link.  Frame synthesis is outside the timed region."""
    import torch.distributed as dist
    import synth_inputs as synth
    from v2ce_toolbox_b200 import dist as vdist

    if world == 1 and not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29541')
        vdist.init_process_group('nccl', device=device, rank=0, world_size=1)
        own_group = True
    else:
        own_group = False
    specs = {
        'long_9000': dict(n=args.long_frames, h=260, w=346, repeat=1, bs=4, kw=dict(infer_type='center', width=346, height=260)),
        'pano_600_2tiles': dict(n=args.pano_frames, h=1080, w=1920, repeat=4, bs=1,
                                kw=dict(infer_type='pano', width=346, height=260)),
        'pano_600_6tiles_h1080': dict(n=args.pano_frames, h=1080, w=1920, repeat=4, bs=1,
                                      kw=dict(infer_type='pano', width=346, height=1080)),
    }
    out = {}
    try:
        for name, sp in specs.items():
            try:
                n = sp['n']
                reader = synth.SynthVideoReader(n, sp['h'], sp['w'], seed=0, repeat=sp['repeat'])
                # materialise this rank's frames up front (synthesis is not part of the workload)
                from v2ce_toolbox_b200 import v2ce as drv
                starts, mode = drv.window_schedule(n, L)
                nb = -(-len(starts) // sp['bs'])
                b0, b1 = vdist.shard_range(nb, world, rank)
                first, count, *_ = vdist.shard_schedule(starts, mode, b0, b1, sp['bs'], L)
                reader.cache_range(first, first + count)
                model = new_model(device)
                common = dict(seq_len=L, batch_size=sp['bs'], fps=30, seed=1, device=device, **sp['kw'])
                # warm-up on a short prefix (first-touch allocations, tensor maps of this geometry, communicators)
                wn = 16 * sp['bs'] * world + 1
                warm = synth.SynthVideoReader(wn, sp['h'], sp['w'], seed=0, repeat=sp['repeat'])
                vdist.stream_clip_sharded(model, warm, wn, world, rank, **common)
                res = {}
                legs = [('device', False, None), ('e2e', True, 'nccl')]
                if world > 1:
                    legs.append(('e2e_shm_merge', True, 'shm'))       # every rank copies its shard into shared memory
                for leg, to_host, merge in legs:
                    # the warmed-up model runs every leg: its runner owns the pinned staging and device buffers (a fresh
                    # model would allocate them inside the timed region); stream_clip_sharded continues the
                    # spectral-norm schedule from clip to clip
                    m = model
                    runs = []
                    for _ in range(2):
                        # twice, the faster run counts (both are listed): the first full-length run of a leg still
                        # sizes the clip-wide buffers and the merge destination (the warm-up clip is one window per rank)
                        ev = None
                        free_device_memory()
                        dist.barrier()
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        ev, n_events = vdist.stream_clip_sharded(m, reader, n, world, rank, to_host=to_host, merge=merge,
                                                                 **common)
                        torch.cuda.synchronize()
                        dist.barrier()
                        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
                        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
                        runs.append(float(dt.item()))
                    best = min(runs)
                    res[leg] = {'s': best, 'pairs_per_s': (n - 1) / best, 'mevents_per_s': n_events / best / 1e6,
                                'runs_s': runs}
                    if to_host and rank == 0:
                        ts = ev['timestamp']
                        step = max(1, len(ts) // 2_000_000)
                        # bins restart every 1/fps/9 inside a frame: frame-to-frame the stream only moves forward
                        res['monotone_frames'] = bool((np.diff(ts[::step]) >= -40000).all()) if len(ts) > 1 else True
                    del ev
                    free_device_memory()
                # `events` is the count of the last run: the spectral-norm power iteration advances with every model call
                # (reference semantics, spectral_norm.py) and the warm-up clip has one window per rank, so the last
                # digits of the count differ from run to run and from N to N; sharded == single-process equality is
                # checked on fresh models (sharded_parity, tests/test_gpu_dist.py)
                res.update({'frames': n, 'pairs': n - 1, 'events': int(n_events), 'stream_bytes': int(n_events) * 13,
                            'source': [sp['h'], sp['w']], 'batch_size': sp['bs'], **{k: v for k, v in sp['kw'].items()}})
                out[name] = res
                del reader, model
            except Exception as e:                      # noqa: BLE001 -- one clip must not take the others down
                out[name] = {'error': f'{type(e).__name__}: {e}'}
                if world > 1:
                    raise                                # ranks would lose step with each other's collectives
            free_device_memory()
    finally:
        if own_group:
            dist.destroy_process_group()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--headline-only', action='store_true', help='skip the secondary records (ef, ldati, library, clips)')
    ap.add_argument('--long-frames', type=int, default=9000)
    ap.add_argument('--pano-frames', type=int, default=600)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the results of the last timed step as DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the results of the CUDA path (--impl ours)')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the V2CE B200 path has no CPU fallback '
                         '(use --impl reference for the CPU oracle arm)')
    if world > 1:
        from v2ce_toolbox_b200 import dist as vdist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        vdist.init_process_group('nccl', device=torch.device('cuda', local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()            # all groups, the host-side gloo group included


if __name__ == '__main__':
    main()
