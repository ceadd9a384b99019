"""GPU parity of the driver level: the drop-in v2ce.py functions and the device-resident CLI path
against the reference's golden voxels and the CPU oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import ef_oracle, pipeline_oracle, synth
from oracle.ref_harness import FakeVideoReader

pytestmark = pytest.mark.gpu


def _model(seed, init='lively'):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(seed, init))
    return m.eval().to('cuda')


@pytest.mark.parametrize('name', ['center', 'pano'])
def test_video_to_voxels_matches_reference_golden(name, golden, golden_meta):
    """Same frames / weights / batching the unmodified reference processed on CPU (tests/golden)."""
    from v2ce_toolbox_b200 import v2ce as drv
    g = golden('pipeline')
    m = golden_meta['pipeline'][name]
    frames = synth.make_video(m['n_frames'], m['H'], m['W'], seed=m['video_seed'])
    vox = drv.video_to_voxels(_model(m['sd_seed'], m['init']), vidcap=FakeVideoReader(frames), infer_type=m['infer_type'],
                              seq_len=16, width=m['width'], height=m['H'], batch_size=m['batch_size'])
    ref = g[f'{name}_voxel']
    assert vox.shape == ref.shape and vox.dtype == np.float32
    rel = np.linalg.norm(vox - ref) / np.linalg.norm(ref)
    from conftest import record_measurement
    record_measurement('pipeline_voxel_vs_reference_golden', name=name, init=m['init'], rel_l2=float(rel))
    assert rel <= 1.6e-2, rel                                 # 'lively' stress weights: see tests/test_gpu_unet.py


@pytest.mark.parametrize('n_frames,bs,seq_len', [pytest.param(20, 2, 16, id='20-2'), pytest.param(33, 1, 16, id='33-1'),
                                                 pytest.param(36, 4, 16, id='36-4'),
                                                 # --seq_len 10 / 8 with the last window pulled back
                                                 pytest.param(26, 2, 10, id='26-2-seq10'),
                                                 pytest.param(21, 3, 8, id='21-3-seq8')])
def test_stream_clip_events_and_frames_bit_exact_on_device_voxels(n_frames, bs, seq_len):
    """The CLI path (voxels never leave the GPU) must produce exactly what the reference's steps produce
    from the same voxels: event frames and the offset, concatenated event stream."""
    _check_stream_clip(n_frames, bs, seq_len=seq_len)


@pytest.mark.parametrize('n_frames,bs', [(16, 1), (2, 1), (3, 2), (17, 4)])
def test_stream_clip_tiny_clips(n_frames, bs):
    """Clips of one window or less: a 16-frame clip's only window starts at frame -1 and keeps 15 pairs (SURVEY.md
    F8a), 2 and 3 frames keep 1 and 2 pairs; the host driver handles them like the reference
    (tests/test_driver_vs_reference_live.py), this is the device-resident path."""
    _check_stream_clip(n_frames, bs)


@pytest.mark.parametrize('n_frames,bs', [(2, 1), (3, 1), (8, 2), (9, 1), (10, 2), (17, 1), (40, 2)])
def test_stream_clip_image_folders_incl_tiny_ones(n_frames, bs, tmp_path):
    """ADVICE round 1: an image folder of <= 16 frames has a negative window start; image_paths[start:] then clamps
    to the frames that exist (a 9-frame folder yields 7 pairs, a 10-frame one 6: the reference's [-mode:] slice keeps
    what is there), and the device-resident path must do what the host driver / the reference do."""
    import cv2
    H, W = 28, 36
    frames = synth.make_video(n_frames, H, W, seed=9)
    paths = []
    for i, f in enumerate(frames):
        paths.append(str(tmp_path / f'{i:04d}.png'))
        cv2.imwrite(paths[-1], f)
    _check_stream_clip(n_frames, bs, image_paths=paths)


def _check_stream_clip(n_frames, bs, image_paths=None, seq_len=16):
    from v2ce_toolbox_b200 import v2ce as drv
    H, W = 28, 36
    frames = synth.make_video(n_frames, H, W, seed=9)
    src = dict(image_paths=image_paths) if image_paths is not None else dict(vidcap=FakeVideoReader(frames))
    vox = drv.video_to_voxels(_model(6), infer_type='center', seq_len=seq_len, width=W, height=H, batch_size=bs, **src)
    vox = vox * np.float32(3)                                 # the check below feeds the same scaled voxels to both sides
    if image_paths is None:
        assert vox.shape[0] == n_frames - 1

    class Scaled(torch.nn.Module):                            # same model, outputs scaled like `vox`
        def __init__(self, inner):
            super().__init__()
            self.inner = inner

        def forward(self, x):
            return self.inner(x) * 3.0

    src = dict(image_paths=image_paths) if image_paths is not None else dict(vidcap=FakeVideoReader(frames))
    res = drv.stream_clip(Scaled(_model(6)), infer_type='center', seq_len=seq_len, width=W,
                          height=H, batch_size=bs, fps=30, ceil=10, upper_bound_percentile=98, seed=77, **src)
    assert res.n_pairs == vox.shape[0]
    want_frames, want_ub, _ = ef_oracle.event_frames_oracle(vox, 10, 98, True)
    assert res.ef_upper_bound == want_ub
    assert np.array_equal(res.ef_frames, want_frames)
    want = pipeline_oracle.event_stream(vox, fps=30, stage2_batch_size=24, seed=77, flavor='cuda')
    assert res.event_stream.dtype.itemsize == 13 and len(res.event_stream) == len(want)
    for f in ('timestamp', 'x', 'y', 'polarity'):
        assert np.array_equal(res.event_stream[f], want[f]), f


def test_cli_writes_reference_named_outputs(tmp_path):
    import cv2
    from v2ce_toolbox_b200 import v2ce as drv
    H, W = 40, 52
    frames = synth.make_video(18, H, W, seed=3)
    folder = tmp_path / 'clip'
    folder.mkdir()
    for i, f in enumerate(frames):
        cv2.imwrite(str(folder / f'{i:04d}.png'), f)
    ckpt = tmp_path / 'w.pt'
    torch.save(synth.make_state_dict(8, 'lively'), ckpt)
    out = tmp_path / 'out'
    drv.main(['-f', str(folder), '-o', str(out), '-m', str(ckpt), '--width', str(W), '--height', str(H), '-b', '2',
              '--seed', '5', '--out_name_suffix', 't'])
    npz = out / 'clip-ceil_10-fps_30-t-events.npz'
    mp4 = out / 'center-clip-ceil_10-fps_30-t-pred_ef_rgb.mp4'
    assert npz.exists() and mp4.exists() and os.path.getsize(mp4) > 0
    ev = np.load(npz)['event_stream']
    assert ev.dtype.names == ('timestamp', 'x', 'y', 'polarity') and ev.dtype.itemsize == 13
    assert ev['x'].max() < W and ev['y'].max() < H and ev['timestamp'].max() < 17 * 33334


def test_sn_replay_makes_sharded_ranks_match_single_process():
    """A rank that starts at batch k must see the model as it is after k calls (SURVEY F3)."""
    m_all, m_shard = _model(11), _model(11)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 1, 16, 2, 20, 28, generator=g).cuda()
    ys = [m_all(x[i]) for i in range(3)]
    m_shard.sn_advance(2)
    y2 = m_shard(x[2])
    assert torch.equal(ys[2], y2)


def test_batch_runner_overlapped_results_match_oracle():
    """runner.BatchRunner (side-stream transfers, double-buffered outputs) returns, for every batch,
    exactly the oracle's events / frames for the voxels the model produced."""
    from v2ce_toolbox_b200.runner import BatchRunner
    from oracle import ldati_oracle as lo
    H, W = 24, 32
    g = torch.Generator().manual_seed(3)
    units = [torch.randn(2, 16, 2, H, W, generator=g).pin_memory() for _ in range(3)]
    m_run, m_ref = _model(12), _model(12)
    runner = BatchRunner(m_run, 'cuda', fps=30, seed=21)
    # slots=2: a batch must be collected before the submit that reuses its slot
    t0 = runner.submit(units[0], pair_base=0)
    t1 = runner.submit(units[1], pair_base=32)
    r0 = runner.wait(t0)
    t2 = runner.submit(units[2], pair_base=64)
    results = [r0, runner.wait(t1), runner.wait(t2)]
    for i, (ev, fr) in enumerate(results):
        vox = (m_ref(units[i].cuda()).cpu().numpy()).reshape(32, 2, 10, H, W)
        want_fr, _, _ = ef_oracle.event_frames_oracle(vox, 10, 98, True)
        assert np.array_equal(fr, want_fr)
        want = lo.sample_voxel_statistical_oracle(vox, fps=30, seed=21, frame_base=32 * i, flavor='cuda')
        for k, r in enumerate(want):
            r['timestamp'] += pipeline_oracle.frame_offset_us(32 * i + k, 30)
        want = np.concatenate(want)
        assert len(ev) == len(want)
        for f in ('timestamp', 'x', 'y', 'polarity'):
            assert np.array_equal(ev[f], want[f]), (i, f)


def test_event_sink_matches_plain_copy():
    """sink.to_host (pinned double buffer + threaded first-touch copies) returns the same bytes as tensor.cpu()."""
    from v2ce_toolbox_b200 import sink
    g = torch.Generator(device='cuda').manual_seed(0)
    for n in (0, 1000, (3 << 20) + 12345):
        t = torch.randint(0, 256, (n,), dtype=torch.uint8, device='cuda', generator=g)
        got = sink.to_host(t, chunk_bytes=1 << 20, workers=4)
        assert got.dtype == np.uint8 and np.array_equal(got, t.cpu().numpy())
