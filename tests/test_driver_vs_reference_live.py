"""The product's host-side driver (v2ce_toolbox_b200/v2ce.py: pre-processing, window schedule, center crop, pano tiles,
batching, merge -- /root/reference/v2ce.py:45-239) against the UNMODIFIED reference driver, live, on CPU.

Both drivers are handed the same stand-in for the network (a cheap deterministic map (b,L,2,H,W) -> (b,L,20,H,W) that
also depends on the call index, like the real model's spectral-norm state) and the same in-memory clip, with
``Tensor.cuda`` shimmed to the identity; every float of the merged voxel grid must agree.  The tests that import
the reference run only where its sources are found (oracle/ref_harness.py, V2CE_REFERENCE_ROOT)."""
import numpy as np
import pytest
import torch

from oracle import ref_harness as rh, synth

needs_reference = pytest.mark.skipif(not rh.available(), reason='the upstream V2CE-Toolbox sources are not found '
                                                                 '(set V2CE_REFERENCE_ROOT)')


class StandIn(torch.nn.Module):
    """Deterministic, position- and call-dependent stand-in for V2ce3d."""

    def __init__(self):
        super().__init__()
        self.calls = 0

    def forward(self, x):
        self.calls += 1
        b, L, c, H, W = x.shape
        assert c == 2
        ramp = torch.arange(20, dtype=torch.float32).view(1, 1, 20, 1, 1) * 0.25
        pos = torch.arange(W, dtype=torch.float32).view(1, 1, 1, 1, W) * 1e-3 + \
            torch.arange(L, dtype=torch.float32).view(1, L, 1, 1, 1) * 1e-2
        return x.repeat_interleave(10, dim=2) * (1.0 + 0.125 * self.calls) + ramp + pos


CASES = [('center', 16, 1, 26, 40, 36),                       # one window starting at frame -1 (SURVEY.md F8a)
         ('center', 2, 1, 26, 40, 36), ('center', 3, 2, 26, 40, 36),
         ('center', 17, 1, 26, 40, 36), ('center', 20, 2, 26, 40, 36), ('center', 33, 1, 26, 40, 36),
         ('center', 36, 4, 26, 40, 36), ('center', 49, 3, 26, 40, 40), ('center', 18, 2, 26, 40, 30),
         ('center', 40, 2, 52, 80, 36),                       # resized 52x80 -> 26x40, then cropped
         ('pano', 18, 1, 26, 52, 20), ('pano', 20, 2, 26, 40, 20), ('pano', 35, 2, 26, 47, 20),
         ('pano', 33, 1, 52, 104, 20)]                        # resized, 3 tiles, the last one pulled back


@needs_reference
@pytest.mark.parametrize('infer_type,n_frames,batch_size,H,W,width', CASES)
def test_video_to_voxels_equals_reference_driver(infer_type, n_frames, batch_size, H, W, width):
    from v2ce_toolbox_b200 import v2ce as drv
    frames = synth.make_video(n_frames, H, W, seed=n_frames)
    height = 26
    with rh.cpu_cuda_shims():
        want = rh.main_module().video_to_voxels(StandIn(), vidcap=rh.FakeVideoReader(frames), infer_type=infer_type,
                                                seq_len=16, width=width, height=height, batch_size=batch_size)
        got = drv.video_to_voxels(StandIn(), vidcap=rh.FakeVideoReader(frames), infer_type=infer_type, seq_len=16,
                                  width=width, height=height, batch_size=batch_size)
    want, got = np.asarray(want), np.asarray(got)
    assert got.shape == want.shape and got.shape[0] == n_frames - 1
    assert np.array_equal(got.astype(np.float32).view(np.uint32), want.astype(np.float32).view(np.uint32))


def test_window_schedule_and_tiles_equal_reference_arithmetic():
    """The closed forms the product uses against the reference's inline arithmetic (v2ce.py:149-154, 103-111)."""
    from v2ce_toolbox_b200 import v2ce as drv
    for n in range(2, 120):
        starts, mode = drv.window_schedule(n, 16)
        sequence_num = int(np.ceil((n - 1) / 16))
        ref = [i * 16 for i in range(sequence_num)]
        if (n - 1) % 16 != 0:
            ref[-1] = ref[-1] - (16 - (n - 1) % 16)
        assert list(starts) == ref and mode == (n - 1) % 16
    for total, width in ((462, 346), (1920, 346), (692, 346), (346, 346), (52, 20), (40, 20), (47, 20)):
        tiles = drv.pano_tiles(total, width)
        assert tiles[0][0] == 0 and tiles[-1][1] == total
        # a remainder of 0 with total % 346 != 0 keeps the whole pulled-back tile (`out[..., -0:]` in the reference,
        # v2ce.py:120-127): the driver comparison above ('pano', 20, 2, 26, 40, 20) covers that quirk end to end
        assert sum((k if k else width) for _, _, k in tiles) == total


def _write_mp4(path, n_frames, H, W, seed=0):
    import cv2
    frames = synth.make_video(n_frames, H, W, seed=seed)
    vw = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*'mp4v'), 30, (W, H))
    for f in frames:
        vw.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    vw.release()
    return frames


@needs_reference
def test_video_reader_equals_reference_reader(tmp_path):
    """scripts/video_reader.py as the CLI uses it (v2ce.py:333-335,170): same frame count and the same gray frames for
    the index patterns the driver issues -- consecutive windows, the one-frame overlap between windows, a pulled-back
    window (a backward seek) -- although this reader decodes consecutive indices sequentially where the reference
    re-seeks before every frame (video_reader.py:307)."""
    import sys
    from v2ce_toolbox_b200.scripts.video_reader import VideoReader
    ref_mod = sys.modules.get('_v2ce_ref.video_reader')
    if ref_mod is None:
        rh.main_module()
        ref_mod = sys.modules['_v2ce_ref.video_reader']
    path = tmp_path / 'clip.mp4'
    _write_mp4(path, 40, 64, 96)
    ours, ref = VideoReader(str(path), color_mode='GRAY'), ref_mod.VideoReader(str(path), color_mode='GRAY')
    assert ours.frame_count == ref.frame_count == 40
    assert (ours.width, ours.height) == (ref.width, ref.height) == (96, 64)
    assert ours.fps == ref.fps
    # range(-1, 16): the only window of a 16-frame clip starts at -1 (SURVEY.md F8a); both readers must resolve the
    # negative seek the same way
    for idx in (range(0, 17), range(16, 33), range(23, 40), range(5, 8), [39], range(0, 40), range(-1, 16)):
        a, b = ours.read_frames_at_indices(idx), ref.read_frames_at_indices(idx)
        assert a.dtype == b.dtype == np.uint8 and a.shape == b.shape == (len(idx), 64, 96)
        assert np.array_equal(a, b), f'indices {list(idx)[:3]}...'
    ours.frame_count = 20                                     # --max_frame_num (v2ce.py:335)
    assert ours.frame_count == 20
    ours.close()


@needs_reference
def test_cli_flags_equal_the_reference_parser():
    """Drop-in boundary (SURVEY.md 8b): every flag of the reference's argparse block (v2ce.py:283-302), with its option
    strings, type, default, nargs and const, exists unchanged in the product's parser; the product adds only --seed."""
    import ast
    import os
    from v2ce_toolbox_b200 import v2ce as drv
    src = open(os.path.join(rh.REF_ROOT, 'v2ce.py')).read()
    ref = {}
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == 'add_argument':
            flags = tuple(a.value for a in node.args if isinstance(a, ast.Constant))
            kw = {}
            for k in node.keywords:
                if k.arg == 'help':
                    continue
                kw[k.arg] = k.value.id if isinstance(k.value, ast.Name) else ast.literal_eval(k.value)
            ref[flags] = kw
    assert len(ref) >= 18
    ours = {tuple(a.option_strings): a for a in drv.build_parser()._actions if a.option_strings and a.dest != 'help'}
    for flags, kw in ref.items():
        assert flags in ours, f'missing flag {flags}'
        a = ours[flags]
        assert a.default == kw.get('default'), (flags, a.default, kw.get('default'))
        want_type = kw.get('type')
        got_type = getattr(a.type, '__name__', None) if a.type is not None else None
        assert got_type == want_type, (flags, got_type, want_type)
        assert a.nargs == kw.get('nargs') and a.const == kw.get('const'), flags
    assert set(ours) - set(ref) == {('--seed',)}


@needs_reference
def test_drop_in_signatures_equal_the_reference():
    """Same names, positional order and defaults for every callable of the boundary (SURVEY.md 8b); the product may add
    keyword-only extensions (seed / frame_base / draws / flavor on sample_voxel_statistical) and nothing else."""
    import inspect
    from v2ce_toolbox_b200 import v2ce as drv
    from v2ce_toolbox_b200.scripts import LDATI as our_ldati
    main, ref_ldati = rh.main_module(), rh.ldati_module()

    def params(fn):
        return [(p.name, p.default) for p in inspect.signature(fn).parameters.values()
                if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]

    for name in ('get_trained_mode', 'image_pre_processing', 'infer_center_image_unit', 'infer_pano_image_unit',
                 'video_to_voxels', 'merge_voxels', 'write_event_frame_video', 'SBool'):
        assert params(getattr(drv, name)) == params(getattr(main, name)), name
    assert params(our_ldati.sample_voxel_statistical) == params(ref_ldati.sample_voxel_statistical)
    extra = [p.name for p in inspect.signature(our_ldati.sample_voxel_statistical).parameters.values()
             if p.kind == p.KEYWORD_ONLY]
    assert extra == ['seed', 'frame_base', 'draws', 'flavor']
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    assert params(V2ce3d.__init__)[1:] == params(rh.V2ce3d().__init__)[1:]
