"""GPU checks of ClipStream: the window-assembly kernel (csrc/frames.cu) equals the oracle byte for byte, and the
streamed events, preview frames, upper bound and pair count equal stream_clip's on the same frames."""
import cv2
import numpy as np
import pytest
import torch

from oracle import frames_oracle, synth
from oracle.ref_harness import FakeVideoReader

pytestmark = pytest.mark.gpu

CV2_CODES = {'bgr': cv2.COLOR_BGR2GRAY, 'rgb': cv2.COLOR_RGB2GRAY, 'bgra': cv2.COLOR_BGRA2GRAY,
             'rgba': cv2.COLOR_RGBA2GRAY}


def _model(seed=6, init='lively'):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(seed, init))
    return m.eval().to('cuda')


def _assemble(frames_dev, slots, color, x0=0, out_width=None):
    from v2ce_toolbox_b200 import frames as fr
    W = frames_dev[0].shape[1]
    n, L1 = np.asarray(slots).shape
    ow = W - x0 if out_width is None else out_width
    out = torch.full((n, L1, frames_dev[0].shape[0], ow), 0xAB, dtype=torch.uint8, device='cuda')   # poisoned
    got = fr.assemble_windows([fr.device_frame(f, color) for f in frames_dev], slots, color, x0, out_width, out=out)
    assert got.data_ptr() == out.data_ptr()
    return got.cpu().numpy()


# ---- the kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('color', ['bgr', 'rgb', 'bgra', 'rgba'])
def test_kernel_converts_every_colour_like_cv2(color):
    c = frames_oracle.COLORS[color][0]
    v = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255] + ([v & 255 ^ 0x5A] if c == 4 else []),
                   -1).astype(np.uint8).reshape(4096, 4096, c)
    got = _assemble([torch.from_numpy(img).cuda()], [[0]], color)[0, 0]
    assert np.array_equal(got, cv2.cvtColor(img, CV2_CODES[color]))


@pytest.mark.parametrize('color', ['gray', 'bgr', 'rgba'])
@pytest.mark.parametrize('H,W,x0,ow', [(1, 1, 0, 1), (7, 13, 0, 13), (5, 31, 3, 17), (260, 346, 0, 346),
                                       (1080, 1920, 1920 // 2 - 173, 346), (3, 5, 4, 1)])
def test_kernel_equals_oracle_on_views_and_crops(color, H, W, x0, ow):
    """Odd widths, 1x1 frames, the center crop, and sources that are crop views with a row pitch above the width or
    (H, W, C) channels-last views of channels-first memory (copied to a usable layout by device_frame)."""
    c = frames_oracle.COLORS[color][0]
    rng = np.random.default_rng(H * 7 + W)
    shape = (H, W) if c == 1 else (H, W, c)
    big = torch.from_numpy(rng.integers(0, 256, (6, H + 3, W + 5) + shape[2:], dtype=np.uint8)).cuda()
    views = [big[i, 1:H + 1, 2:W + 2] for i in range(6)]                # row pitch (W + 5) * C
    assert views[0].stride(0) == (W + 5) * c
    slots = [[0, 1, 2], [2, 3, 4], [4, 5, 0]]
    want = frames_oracle.assemble_windows([v.cpu().numpy() for v in views], slots, color, x0, ow)
    assert np.array_equal(_assemble(views, slots, color, x0, ow), want)
    if c > 1:                                                           # channels-last view of (C, H, W) memory
        planar = [torch.from_numpy(np.ascontiguousarray(v.cpu().numpy().transpose(2, 0, 1))).cuda().permute(1, 2, 0)
                  for v in views]
        assert np.array_equal(_assemble(planar, slots, color, x0, ow), want)


# ---- ClipStream against stream_clip ------------------------------------------------------------------------------------
def _stream_clip(frames_gray, model=None, **kw):
    from v2ce_toolbox_b200 import v2ce as drv
    res = drv.stream_clip(model or _model(), vidcap=FakeVideoReader(frames_gray), events_to_host=False, **kw)
    if res.event_stream_dev is not None:                 # a view of the runner's buffer, which the next clip reuses
        res.event_stream_dev = res.event_stream_dev.clone()
    return res


def _clip_stream(frames, pushes, model=None, device_frames=True, **kw):
    """Push `frames` in chunks of the sizes `pushes` cycles through; returns (result, batches in order)."""
    from v2ce_toolbox_b200 import ClipStream
    src = torch.from_numpy(frames).cuda() if device_frames else frames
    batches = []
    with ClipStream(model or _model(), **kw) as cs:
        a, k = 0, 0
        while a < len(frames):
            n = pushes[k % len(pushes)]
            batches += cs.push(src[a:a + n])
            a, k = a + n, k + 1
        res = cs.close()
    return res, batches + res.batches


def _assert_same(ref, res, batches, pair_base=0):
    assert res.n_pairs == ref.n_pairs
    assert res.ef_upper_bound == ref.ef_upper_bound
    assert (res.ef_frames is None) == (ref.ef_frames is None)
    if ref.ef_frames is not None:
        assert np.array_equal(res.ef_frames, ref.ef_frames)
    off, pair = 0, pair_base
    stream = ref.event_stream_dev if ref.event_stream_dev is not None else torch.empty(0, dtype=torch.uint8, device='cuda')
    for b in batches:
        assert b.pair_range[0] == pair
        pair = b.pair_range[1]
        n = b.events_dev.numel()
        assert torch.equal(b.events_dev, stream[off:off + n]), (b.pair_range, n)
        off += n
    assert off == stream.numel() and pair - pair_base == ref.n_pairs


def test_benchmark_clip_from_device_and_host_frames():
    """321 frames of 346 x 260 at -b 4, the benchmark's shape: CUDA frames in uneven pushes, host frames one by one."""
    frames = synth.make_video(321, 260, 346, seed=1)
    kw = dict(seq_len=16, width=346, height=260, batch_size=4, fps=30, seed=3)
    ref = _stream_clip(frames, **kw)
    assert ref.n_pairs == 320 and ref.n_events > 0
    _assert_same(ref, *_clip_stream(frames, [5, 40, 1, 97], **kw))
    _assert_same(ref, *_clip_stream(frames, [1], device_frames=False, **kw))


@pytest.mark.parametrize('n_frames', [17, 18, 33, 34, 70])
@pytest.mark.parametrize('seq_len,bs', [(16, 2), (10, 3)])
def test_frame_counts_and_pushes(n_frames, seq_len, bs):
    frames = synth.make_video(n_frames, 28, 36, seed=n_frames)
    kw = dict(seq_len=seq_len, width=36, height=28, batch_size=bs, fps=30, seed=5)
    ref = _stream_clip(frames, **kw)
    for pushes in ([1], [3, 17], [n_frames]):
        _assert_same(ref, *_clip_stream(frames, pushes, **kw))


@pytest.mark.parametrize('infer_type,width', [('center', 36), ('pano', 20)])
def test_resize_route(infer_type, width):
    frames = synth.make_video(37, 60, 112, seed=4)                       # 60 x 112 -> 28 x 52 on the device
    kw = dict(infer_type=infer_type, seq_len=16, width=width, height=28, batch_size=2, fps=30, seed=3)
    ref = _stream_clip(frames, **kw)
    _assert_same(ref, *_clip_stream(frames, [7], **kw))


def test_pano_1080p():
    frames = synth.make_video(20, 1080, 1920, seed=2)
    kw = dict(infer_type='pano', seq_len=16, width=346, height=260, batch_size=1, fps=30, seed=1)
    ref = _stream_clip(frames, **kw)
    assert ref.n_pairs == 19
    _assert_same(ref, *_clip_stream(frames, [6], **kw))


@pytest.mark.parametrize('color', ['bgr', 'rgb', 'bgra', 'rgba'])
def test_colour_device_frames(color):
    """Colour frames pushed to the device equal stream_clip on the frames cv2 converts to gray."""
    c = frames_oracle.COLORS[color][0]
    rng = np.random.default_rng(c)
    col = rng.integers(0, 256, (35, 28, 36, c), dtype=np.uint8)
    col[..., 1] = synth.make_video(35, 28, 36, seed=8)                  # structure the model reacts to
    gray = np.stack([cv2.cvtColor(f, CV2_CODES[color]) for f in col])
    kw = dict(seq_len=16, width=36, height=28, batch_size=2, fps=30, seed=9)
    ref = _stream_clip(gray, **kw)
    _assert_same(ref, *_clip_stream(col, [4], color=color, **kw))


def test_pair_base_and_options():
    frames = synth.make_video(50, 28, 36, seed=12)
    kw = dict(seq_len=16, width=36, height=28, batch_size=2, fps=24, seed=2, pair_base=1000, ceil=5,
              upper_bound_percentile=90, keep_polarity=False)
    ref = _stream_clip(frames, **kw)
    _assert_same(ref, *_clip_stream(frames, [9], **kw), pair_base=1000)
    kw['write_event_frames'] = False
    ref = _stream_clip(frames, **kw)
    assert ref.ef_frames is None
    _assert_same(ref, *_clip_stream(frames, [9], **kw), pair_base=1000)


@pytest.mark.parametrize('n_frames', [2, 3, 9, 10, 16])
def test_short_clips_equal_an_image_list(n_frames, tmp_path):
    """Clips of at most seq_len frames: stream_clip on an image list (a negative first start clamps the slice); a
    16-frame list has a one-frame window and fails, and ClipStream fails the same way."""
    from v2ce_toolbox_b200 import v2ce as drv
    frames = synth.make_video(n_frames, 28, 36, seed=9)
    paths = []
    for i, f in enumerate(frames):
        paths.append(str(tmp_path / f'{i:04d}.png'))
        cv2.imwrite(paths[-1], f)
    kw = dict(seq_len=16, width=36, height=28, batch_size=2, fps=30, seed=4)
    try:
        ref = drv.stream_clip(_model(), image_paths=paths, events_to_host=False, **kw)
    except Exception as e:                                             # noqa: BLE001
        with pytest.raises(type(e)) as got:
            _clip_stream(frames, [1], **kw)
        assert str(got.value) == str(e)
        assert n_frames == 16
        return
    _assert_same(ref, *_clip_stream(frames, [1], **kw))


def test_model_reuse_after_a_stream():
    """ClipStream then stream_clip on model A equals two stream_clip calls on an identically built model B: the
    stream advances the spectral-norm state exactly as a stream_clip call does and leaves the runner reusable."""
    from v2ce_toolbox_b200 import v2ce as drv
    frames = synth.make_video(40, 28, 36, seed=3)
    kw = dict(seq_len=16, width=36, height=28, batch_size=2, fps=30, seed=6)
    a, b = _model(), _model()
    ref1 = _stream_clip(frames, model=b, **kw)
    ref2 = _stream_clip(frames, model=b, **kw)
    _assert_same(ref1, *_clip_stream(frames, [11], model=a, **kw))
    got2 = _stream_clip(frames, model=a, **kw)
    assert torch.equal(got2.event_stream_dev, ref2.event_stream_dev)
    assert np.array_equal(got2.ef_frames, ref2.ef_frames) and got2.ef_upper_bound == ref2.ef_upper_bound
    from v2ce_toolbox_b200 import ClipStream
    with pytest.raises(RuntimeError, match='already converting'):
        with ClipStream(a):
            drv.stream_clip(a, vidcap=FakeVideoReader(frames), **kw)


def test_device_memory_is_bounded():
    """A 2 000-frame stream with write_event_frames=False: once the allocator has seen its first batches, the peak does
    not grow with the frame count."""
    from v2ce_toolbox_b200 import ClipStream
    # 64 frames = one batch of four 16-pair windows: every batch sees the same frames, so a growing peak is the stream's
    pool = torch.from_numpy(synth.make_video(64, 260, 346, seed=5)).cuda()
    peaks = []
    n_pairs = 0
    with ClipStream(_model(), seq_len=16, width=346, height=260, batch_size=4, write_event_frames=False) as cs:
        for a in range(0, 2000, 16):
            for b in cs.push(pool[a % 64:a % 64 + 16]):
                n_pairs += b.pair_range[1] - b.pair_range[0]
            b = None
            if a % 320 == 0 and a > 0:
                torch.cuda.synchronize()
                if a == 320:
                    torch.cuda.reset_peak_memory_stats()
                else:
                    peaks.append(torch.cuda.max_memory_allocated())
        res = cs.close()
    assert res.n_pairs == 1999 and res.ef_frames is None
    assert n_pairs + sum(b.pair_range[1] - b.pair_range[0] for b in res.batches) == 1999
    from conftest import record_measurement
    record_measurement('clip_stream_peak_bytes', peaks=peaks)
    assert len(peaks) == 5 and peaks[-1] <= peaks[0] * 1.02 + (64 << 20), peaks
