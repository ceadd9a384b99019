"""CPU checks of ClipStream: its batch schedule equals stream_clip's for every way frames arrive, the colour oracle equals
the installed OpenCV over all 2^24 colours, and argument errors are raised before any device work."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import frames_oracle
from oracle.ref_harness import FakeVideoReader
from v2ce_toolbox_b200 import clip_stream as cs_mod
from v2ce_toolbox_b200 import v2ce as drv


class _NoModel:
    """Stands in for a model: no forward_frames, so frames of any size take the device-resize route."""


def _stream_clip_batches(n_frames, seq_len, batch_size, pair_base):
    """stream_clip's submissions for an image list of n_frames frames, as its loop made them before ClipStream existed:
    windows in schedule order, `batch_size` per batch, the last batch trimmed to `mode` pairs, pair indices counted the
    way BatchRunner.submit counts them."""
    starts, mode = drv.window_schedule(n_frames, seq_len)
    out, pending, pair = [], [], pair_base
    for i, s in enumerate(starts):
        pending.append(list(range(n_frames)[int(s):int(s) + seq_len + 1]))
        is_last = i == len(starts) - 1
        if len(pending) == batch_size or is_last:
            trim = mode if (is_last and mode != 0) else 0
            out.append((pending, trim, pair))
            L = len(pending[0]) - 1
            pair += (len(pending) - 1) * L + (min(trim, L) if trim else L)
            pending = []
    return out, pair - pair_base


class _Recording(cs_mod.ClipStream):
    """A ClipStream whose device half is a stand-in runner: it records what would be submitted."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.submitted, self.pair = [], self.pair_base

    def _run(self, windows, trim):
        frames = [list(w) for w in windows]
        assert all(i in self._ring for w in frames for i in w), 'a frame a batch needs has left the ring'
        assert len(self._ring) <= (self.schedule.batch_size + 1) * self.schedule.seq_len + 1
        self.submitted.append((frames, trim, self.pair))
        L = len(frames[0]) - 1
        self.pair += (len(frames) - 1) * L + (min(trim, L) if trim else L)
        return []


@pytest.mark.parametrize('seq_len', [8, 10, 16])
@pytest.mark.parametrize('push', [1, 3, 17, None])
def test_schedule_equals_stream_clip_batching(seq_len, push):
    video = np.arange(70, dtype=np.uint8).reshape(70, 1, 1) * np.ones((1, 2, 3), np.uint8)
    for batch_size in range(1, 6):
        for n_frames in range(1, 71):
            s = _Recording(_NoModel(), seq_len=seq_len, batch_size=batch_size, pair_base=5)
            step = push or n_frames
            for a in range(0, n_frames, step):
                s.push(video[a:min(a + step, n_frames)])
            res = s.close()
            want, n_pairs = _stream_clip_batches(n_frames, seq_len, batch_size, 5)
            assert s.submitted == want, (n_frames, batch_size)
            assert res.n_pairs == 0 and res.batches == []          # the stand-in hands nothing out
            assert s.pair - 5 == n_pairs


def test_empty_stream_fails_like_stream_clip_on_an_empty_list():
    with pytest.raises(IndexError) as want:
        drv.stream_clip(_NoModel(), image_paths=[])
    s = cs_mod.ClipStream(_NoModel())
    with pytest.raises(IndexError) as got:
        s.close()
    assert str(got.value) == str(want.value)


def test_one_frame_gives_the_empty_result_of_stream_clip():
    s = cs_mod.ClipStream(_NoModel())
    assert s.push(np.zeros((1, 4, 6), np.uint8)) == []
    res = s.close()
    assert (res.batches, res.ef_frames, res.ef_upper_bound, res.n_pairs) == ([], None, None, 0)


@pytest.mark.parametrize('color', ['bgr', 'rgb', 'bgra', 'rgba'])
def test_colour_oracle_equals_cv2_for_every_colour(color):
    import cv2
    v = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    if color in ('bgra', 'rgba'):
        alpha = (np.arange(1 << 24, dtype=np.uint32) * 2654435761 >> 24).astype(np.uint8).reshape(4096, 4096, 1)
        img = np.concatenate([img, alpha], axis=-1)                # alpha must not matter
    code = {'bgr': cv2.COLOR_BGR2GRAY, 'rgb': cv2.COLOR_RGB2GRAY, 'bgra': cv2.COLOR_BGRA2GRAY,
            'rgba': cv2.COLOR_RGBA2GRAY}[color]
    assert np.array_equal(frames_oracle.to_gray(img, color), cv2.cvtColor(img, code))


def test_oracle_window_gather_and_crop():
    rng = np.random.default_rng(1)
    fr = rng.integers(0, 256, (5, 6, 9, 3), dtype=np.uint8)
    got = frames_oracle.assemble_windows(fr, [[0, 1, 2], [2, 3, 4]], 'rgb', x0=2, out_width=4)
    assert got.shape == (2, 3, 6, 4)
    assert np.array_equal(got[1, 0], got[0, 2])
    assert np.array_equal(got[1, 2], frames_oracle.to_gray(fr[4], 'rgb')[:, 2:6])


def test_argument_errors():
    g = np.zeros((1, 6, 8), np.uint8)                              # one frame: close() has no batch to run
    s = cs_mod.ClipStream(_NoModel(), seq_len=4)
    s.push(g)
    with pytest.raises(ValueError, match='shape'):
        s.push(np.zeros((1, 6, 10), np.uint8))                     # another resolution
    with pytest.raises(ValueError, match='uint8'):
        s.push(g.astype(np.float32))
    with pytest.raises(ValueError, match='uint8'):
        s.push(torch.zeros(1, 6, 8, dtype=torch.int16))
    with pytest.raises(ValueError, match='gray frames'):
        s.push(np.zeros((1, 6, 8, 3), np.uint8))                   # colour in a gray stream
    s.close()
    with pytest.raises(RuntimeError, match='after close'):
        s.push(g)
    with pytest.raises(RuntimeError, match='called already'):
        s.close()

    with cs_mod.ClipStream(_NoModel(), color='bgra') as c:
        with pytest.raises(ValueError, match='bgra frames'):
            c.push(np.zeros((1, 6, 8, 3), np.uint8))               # three channels in a four-channel stream
        with pytest.raises(ValueError, match='fewer than 2 rows'):
            c.push(np.zeros((1, 1, 8, 4), np.uint8))
    with pytest.raises(ValueError, match='color'):
        cs_mod.ClipStream(_NoModel(), color='hsv')
    with pytest.raises(ValueError, match='infer_type'):
        cs_mod.ClipStream(_NoModel(), infer_type='left')


def test_one_open_stream_per_model():
    m = _NoModel()
    a = cs_mod.ClipStream(m)
    with pytest.raises(RuntimeError, match='already converting'):
        cs_mod.ClipStream(m)
    with pytest.raises(RuntimeError, match='already converting'):
        drv.stream_clip(m, vidcap=FakeVideoReader(np.zeros((40, 4, 4), np.uint8)))
    with cs_mod.ClipStream(_NoModel()):                            # another model is free
        pass
    a.push(np.zeros((1, 4, 4), np.uint8))
    a.close()
    with cs_mod.ClipStream(m) as c:                                # closed: the model is free again; left without
        c.push(np.zeros((3, 4, 4), np.uint8))                      # close(), it is freed as well
    with pytest.raises(IndexError):
        cs_mod.ClipStream(m).close()                               # an empty clip fails like stream_clip's, and frees it
    cs_mod.ClipStream(m).__exit__(None, None, None)


def test_assemble_windows_argument_checks_run_without_a_gpu():
    from v2ce_toolbox_b200 import _lib
    lib = _lib.load()
    tab, slots, out = (ctypes.c_int64 * 2)(), (ctypes.c_int32 * 1)(), (ctypes.c_uint8 * 16)()
    assert lib.v2ce_assemble_windows(None, slots, 1, 1, 4, 4, 1, 0, 0, 4, out, None) != 0
    assert b'NULL' in lib.v2ce_last_error()
    assert lib.v2ce_assemble_windows(tab, slots, 1, 1, 4, 4, 2, 0, 0, 4, out, None) != 0
    assert b'channels' in lib.v2ce_last_error()
    assert lib.v2ce_assemble_windows(tab, slots, 1, 1, 4, 4, 3, 2, 0, 4, out, None) != 0
    assert b'rgb_order' in lib.v2ce_last_error()
    assert lib.v2ce_assemble_windows(tab, slots, 1, 1, 4, 4, 1, 0, 1, 4, out, None) != 0
    assert b'outside' in lib.v2ce_last_error()
    assert lib.v2ce_assemble_windows(tab, slots, 0, 1, 4, 4, 1, 0, 0, 4, out, None) != 0
    assert b'window table' in lib.v2ce_last_error()
