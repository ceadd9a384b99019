"""Drop-in for /root/reference/v2ce.py: same CLI flags, function names, arguments and output
files, with the device work routed through libv2ce_b200.so.

Two ways in:
  * the reference's functions, one for one (``get_trained_mode``, ``image_pre_processing``,
    ``infer_center_image_unit``, ``infer_pano_image_unit``, ``video_to_voxels``, ``merge_voxels``,
    ``write_event_frame_video``) -- same inputs, same host-side return values;
  * ``stream_clip`` (what ``main`` uses): the reference's __main__ (v2ce.py:322-372) re-scheduled
    so voxels never leave the GPU.  Per batch of windows: H2D image units -> UNet -> event-frame
    sums + LDATI on the device -> packed events D2H.  The clip-global percentile of the preview
    video (v2ce.py:262-264) is taken at the end over the (N,2,H,W) sums kept on the device.
    Outputs are identical to running the reference's steps in its own order, because windows,
    frame pairs and pano tiles are independent and the uniform draws are a counter-based
    function of the global frame index (SURVEY.md F7).
"""
import argparse
import logging
import os
import os.path as op
from functools import partial
from pathlib import Path

import numpy as np
import torch

from . import event_frames as _ef
from . import ldati as _ldati
from ._lib import V2ceError
from .scripts.LDATI import sample_voxel_statistical
from .scripts.v2ce_3d import V2ce3d

logger = logging.getLogger('V2CE')


def SBool(v):
    if isinstance(v, bool):
        return v
    if v.lower() in ('yes', 'true', 't', 'y', '1'):
        return True
    if v.lower() in ('no', 'false', 'f', 'n', '0'):
        return False
    raise argparse.ArgumentTypeError('Boolean value expected.')


def get_trained_mode(model_path='./weights/v2ce_3d.pt'):
    """v2ce.py:30-43 -- load the checkpoint into the B200 model."""
    model = V2ce3d()
    model.load_state_dict(torch.load(model_path, map_location='cpu'))
    model = model.eval()
    model = model.to('cuda')
    return model


def image_pre_processing(images, height=260):
    """v2ce.py:45-64 -- (N,H,W) uint8 gray frames -> (N-1,2,H',W') float32 image units.
    /255, bilinear resize to `height`, pair stacking, Normalize(0.153, 0.165)."""
    import cv2
    images = images.astype(np.float32) / 255
    images = np.stack([cv2.resize(img, (int(img.shape[1] / img.shape[0] * height), height)) for img in images], axis=0)
    units = np.stack([images[:-1], images[1:]], axis=1)
    units = (units - np.float32(0.153)) / np.float32(0.165)
    return torch.from_numpy(np.ascontiguousarray(units, dtype=np.float32))


def window_schedule(frame_count, seq_len=16):
    """v2ce.py:149-154 -- window starts; the last one is pulled back when (F-1) % seq_len != 0."""
    sequence_num = int(np.ceil((frame_count - 1) / seq_len))
    mode = (frame_count - 1) % seq_len
    starts = np.arange(sequence_num) * seq_len
    if mode != 0:
        starts[-1] -= (seq_len - mode)
    return starts, mode


def batch_plan(starts, mode, batch_size):
    """v2ce.py:158-176 batching of the windows `starts`: [(first window, end window, trim_last_window_to)], `batch_size`
    consecutive windows per model call; the batch holding the last window keeps only the last `mode` pairs of it
    (v2ce.py:227-236, BatchRunner.submit)."""
    n = len(starts)
    return [(a, min(a + batch_size, n), mode if a + batch_size >= n else 0) for a in range(0, n, batch_size)]


def pano_tiles(total_width, width=346):
    """v2ce.py:103-111 -- (src_start, src_end, columns kept from the right) per 346-px tile."""
    n = int(np.ceil(total_width / width))
    exact = total_width % 346 == 0            # the reference tests the literal 346 here
    rem = total_width % width
    tiles = []
    for i in range(n):
        if i == n - 1 and not exact:
            tiles.append((total_width - width, total_width, rem))
        else:
            tiles.append((i * width, (i + 1) * width, width))
    return tiles


@torch.no_grad()
def _center_device(model, image_units, width=346):
    c = image_units.shape[-1] // 2
    units = image_units[..., c - width // 2:c + width // 2]
    return model(units.float().contiguous().cuda(non_blocking=True))


@torch.no_grad()
def _pano_device(model, image_units, width=346):
    parts = []
    for (a, b, keep) in pano_tiles(image_units.shape[-1], width):
        out = model(image_units[..., a:b].float().contiguous().cuda(non_blocking=True))
        parts.append(out[..., -keep:] if keep != width else out)
    return torch.cat(parts, dim=-1) if len(parts) > 1 else parts[0]


@torch.no_grad()
def infer_center_image_unit(model, image_units, width=346):
    """v2ce.py:66-89 -- center crop, model, back to host."""
    return _center_device(model, image_units, width).cpu()


@torch.no_grad()
def infer_pano_image_unit(model, image_units, width=346):
    """v2ce.py:91-129 -- 346-px width tiles (one model call each), concatenated on the width."""
    return _pano_device(model, image_units, width).cpu()


class FramePrefetcher:
    """Decodes the frames of an image folder ahead of the device pipeline (SURVEY.md N1: at GPU speed the serial
    ``cv2.imread`` loop of v2ce.py:158-166 is the bottleneck of a clip).  Frames are decoded once each on a thread pool
    (OpenCV releases the GIL), `lookahead` windows beyond the one being consumed; ``window(start, seq_len)`` returns the
    same (seq_len+1, H, W) uint8 stack the serial loop builds."""

    def __init__(self, image_paths, starts, seq_len, lookahead=8, workers=8):
        from concurrent.futures import ThreadPoolExecutor
        self.paths = image_paths
        self.starts = [int(s) for s in starts]
        self.seq_len = seq_len
        self.lookahead = lookahead
        self.pool = ThreadPoolExecutor(max_workers=workers)
        self.futures = {}
        self.next_window = 0

    @staticmethod
    def _decode(path):
        import cv2
        img = cv2.imread(path, cv2.IMREAD_GRAYSCALE)
        if img is None:
            raise FileNotFoundError(f'cv2.imread could not read {path}')
        return img

    def _submit_through(self, k):
        while self.next_window <= min(k, len(self.starts) - 1):
            st = self.starts[self.next_window]
            for i in range(st, min(st + self.seq_len + 1, len(self.paths))):
                if i not in self.futures:
                    self.futures[i] = self.pool.submit(self._decode, self.paths[i])
            self.next_window += 1

    def window(self, k):
        """Frames of the k-th scheduled window; windows must be requested in schedule order."""
        self._submit_through(k + self.lookahead)
        st = self.starts[k]
        frames = [self.futures[i].result() for i in range(st, min(st + self.seq_len + 1, len(self.paths)))]
        for i in [i for i in self.futures if i < st]:         # windows only move forward (the pulled-back last one
            del self.futures[i]                               # starts inside the one before it)
        return np.stack(frames, axis=0)

    def close(self):
        self.pool.shutdown(wait=False, cancel_futures=True)


def _read_window(image_paths, vidcap, start, seq_len):
    import cv2
    idx = range(start, start + seq_len + 1)
    if vidcap is not None:
        return vidcap.read_frames_at_indices(idx)
    return np.stack([cv2.imread(p, cv2.IMREAD_GRAYSCALE) for p in image_paths[start:start + seq_len + 1]], axis=0)


def _window_reader(image_paths, vidcap, starts, seq_len):
    """k -> frames of the k-th window: prefetched decode for image folders, the reader's own access otherwise."""
    ascending = all(int(a) <= int(b) for a, b in zip(starts[:-1], starts[1:]))
    if vidcap is None and len(starts) > 1 and int(starts[0]) >= 0 and ascending:
        pf = FramePrefetcher(image_paths, starts, seq_len)
        return pf.window, pf.close
    return (lambda k: _read_window(image_paths, vidcap, int(starts[k]), seq_len)), (lambda: None)


def _background(gen, depth=2):
    """Run the batch generator `gen` on a producer thread, `depth` batches ahead of the consumer: decoding, cv2.resize
    and batch assembly (all of which release the GIL) then overlap the consumer's CUDA submissions and waits instead of
    alternating with them.  Items arrive in order; an exception in the producer is re-raised at the consumer; closing the
    consumer early stops the producer."""
    import queue
    import threading
    q = queue.Queue(maxsize=depth)
    end, stop = object(), threading.Event()

    def put(item):
        while not stop.is_set():
            try:
                q.put(item, timeout=0.05)
                return True
            except queue.Full:
                pass
        return False

    def produce():
        try:
            for item in gen:
                if not put(item):
                    break
            else:
                put(end)
        except BaseException as e:                      # noqa: B902 -- handed to the consumer
            put(e)
        finally:
            gen.close()

    th = threading.Thread(target=produce, name='v2ce-batches', daemon=True)
    th.start()
    try:
        while True:
            item = q.get()
            if item is end:
                return
            if isinstance(item, BaseException):
                raise item
            yield item
    finally:
        stop.set()
        th.join(timeout=5.0)


def _batches(image_paths, vidcap, seq_len, height, batch_size, schedule=None):
    """Yield (image_units (b,L,2,H',W') float32 host tensor, is_last) in the reference's batching.
    `schedule` = (window starts, mode) overrides the schedule derived from the frame count (a rank's share of a clip)."""
    frame_count = vidcap.frame_count if vidcap is not None else len(image_paths)
    starts, mode = schedule if schedule is not None else window_schedule(frame_count, seq_len)
    read, close = _window_reader(image_paths, vidcap, starts, seq_len)
    try:
        for a, e, _trim in batch_plan(starts, mode, batch_size):
            pending = [image_pre_processing(read(i), height)[None] for i in range(a, e)]
            yield (torch.cat(pending, dim=0) if len(pending) > 1 else pending[0]), e == len(starts)
    finally:
        close()


@torch.no_grad()
def video_to_voxels(model, image_paths=None, vidcap=None, infer_type='center', seq_len=16, width=346, height=260,
                    batch_size=1):
    """v2ce.py:131-209 -- returns the host voxel grid (N,2,10,H,W) float32 like the reference."""
    assert image_paths is not None or vidcap is not None
    frame_count = vidcap.frame_count if vidcap is not None else len(image_paths)
    _, mode = window_schedule(frame_count, seq_len)
    outs = []
    out_width = width
    for units, _last in _batches(image_paths, vidcap, seq_len, height, batch_size):
        if infer_type == 'center':
            out_width = width
            pred = infer_center_image_unit(model, units, width)
        elif infer_type == 'pano':
            out_width = units.shape[-1]
            pred = infer_pano_image_unit(model, units, width)
        else:
            raise ValueError(f'Invalid infer_type {infer_type}')
        outs.append(pred.numpy())
    return merge_voxels(outs, height=height, width=out_width, mode=mode)


def merge_voxels(voxel_list, height=260, width=346, mode=0):
    """v2ce.py:211-239 -- (b,L,20,H,W) batches -> (N,2,10,H,W); the pulled-back last window keeps its last `mode` pairs."""
    chunks = [v.reshape(-1, 2, 10, height, width) for v in voxel_list[:-1]]
    last = voxel_list[-1]
    if last.shape[0] > 1:
        chunks.append(last[:-1].reshape(-1, 2, 10, height, width))
    tail = last[-1][-mode:] if mode != 0 else last[-1]
    chunks.append(tail.reshape(-1, 2, 10, height, width))
    return np.concatenate(chunks, axis=0)


write_event_frame_video = _ef.write_event_frame_video      # v2ce.py:241-280


def frame_offset_us(i, fps):
    """v2ce.py:365 -- Python double arithmetic, then int()."""
    return int(i * 1 / fps * 1e6)


class ClipResult:
    def __init__(self, event_stream, ef_frames, ef_upper_bound, n_pairs):
        self.event_stream = event_stream
        self.ef_frames = ef_frames
        self.ef_upper_bound = ef_upper_bound
        self.n_pairs = n_pairs
        self.event_stream_dev = None
        self.ef_sums_dev = None            # (n_pairs, 2 | 1, H, W) float32 per-pair sums (keep_event_frame_sums=True)
        self.n_events = 0 if event_stream is None else len(event_stream)


def _window_batches_u8(image_paths, vidcap, seq_len, batch_size, schedule, width):
    """Raw uint8 windows in the reference's batching: (b, L+1, H, width) center-cropped like v2ce.py:78, or the whole
    frames (b, L+1, H, W) when `width` is None (the device then resizes them, preprocess.image_units_device)."""
    frame_count = vidcap.frame_count if vidcap is not None else len(image_paths)
    starts, mode = schedule if schedule is not None else window_schedule(frame_count, seq_len)
    read, close = _window_reader(image_paths, vidcap, starts, seq_len)
    pin = torch.cuda.is_available()
    try:
        for a, e, _trim in batch_plan(starts, mode, batch_size):
            pending = []
            for i in range(a, e):
                fr = np.asarray(read(i))
                if width is not None:
                    c = fr.shape[-1] // 2
                    fr = fr[..., c - width // 2:c + width // 2]
                pending.append(fr)
            # ONE copy per frame, straight into the page-locked batch the H2D transfer reads (a 1080p window is
            # 35 MB: stacking, concatenating and pinning it separately made the host the bottleneck of a pano clip)
            out = torch.empty((len(pending),) + tuple(pending[0].shape), dtype=torch.uint8, pin_memory=pin)
            o = out.numpy()
            for j, w in enumerate(pending):
                np.copyto(o[j], w)
            yield out, e == len(starts)
    finally:
        close()


def _frame_route(model, infer_type, dtype, shape, height, width, device_resize, pano=_pano_device):
    """How the gray frames of a clip, `shape` (..., H, W), reach the model: ('native', None) when they already have the
    model's resolution (raw uint8 windows, center-cropped, go to forward_frames; the resize of image_pre_processing is
    the identity and the rest of it runs inside the head conv); ('raw', infer) for uint8 frames at another resolution
    (whole uint8 windows are uploaded; /255, the cv2-exact bilinear resize, pair stacking and Normalize run in one
    kernel, preprocess.image_units_device, bit-identical to the host path -- SURVEY.md N1); (None, None) otherwise
    (float image units from the host)."""
    H, W = shape[-2], shape[-1]
    if (infer_type == 'center' and hasattr(model, 'forward_frames') and dtype == np.uint8 and H == height and
            int(W / H * height) == W and W >= width and width % 2 == 0):
        return 'native', None
    if device_resize and dtype == np.uint8 and len(shape) == 3 and H >= 2:
        from .preprocess import image_units_device
        tile = _center_device if infer_type == 'center' else pano
        return 'raw', (lambda u8: tile(model, image_units_device(u8, height), width))
    return None, None


def _claim_model(model):
    """One clip at a time per model: the spectral-norm state advances per model call, so two interleaved clips would
    each change the other's sigma, and they would share the model's BatchRunner."""
    if model.__dict__.get('_v2ce_clip_open'):
        raise RuntimeError('this model is already converting a clip (a ClipStream that has not been closed)')
    model.__dict__['_v2ce_clip_open'] = True


def _release_model(model):
    model.__dict__['_v2ce_clip_open'] = False


class _ClipRun:
    """The device half of one clip, shared by stream_clip and clip_stream.ClipStream: the model's BatchRunner, the pair
    index each batch starts at, and the clip-global event frames (v2ce.py:262-264) over the per-pair sums.
    hand_out=False collects the events of every batch in one device buffer (runner.collected_events); True gives each
    batch's events a tensor of its own (Ticket.events_out)."""

    def __init__(self, model, device, infer, fps, ceil, percentile, keep_polarity, seed, pair_base, keep_sums,
                 hand_out, clip_pairs=0):
        from .runner import BatchRunner
        # the runner owns ~0.5 GB of pinned staging buffers whose allocation costs more than a short clip's compute:
        # one per (model, device), reused across calls
        cache = model.__dict__.setdefault('_v2ce_runners', {})
        runner = cache.get(str(device))
        if runner is None:
            runner = cache[str(device)] = BatchRunner(model, device, per_batch_frames=False, copy_out=False,
                                                      collect_on_device=True)
        runner.fps, runner.ceil, runner.percentile, runner.keep, runner.seed = fps, ceil, percentile, keep_polarity, seed
        runner.infer = infer
        runner.collect_on_device, runner.events_out = not hand_out, hand_out
        runner.sums = []
        runner.reset_collection()
        runner.clip_pairs = clip_pairs
        self.runner, self.device, self.keep_sums = runner, device, keep_sums
        self.percentile, self.ceil, self.keep = percentile, ceil, keep_polarity
        self.pair_idx = pair_base

    def submit(self, x, trim_last_window_to):
        t = self.runner.submit(x, self.pair_idx, keep_sums=self.keep_sums, trim_last_window_to=trim_last_window_to)
        self.pair_idx += t.n_pairs
        return t

    def event_frames(self, write_event_frames):
        """(uint8 BGR preview frames | None, upper bound | None, per-pair sums | None) once every batch is submitted."""
        frames, ub, sums = None, None, None
        if self.keep_sums:
            torch.cuda.current_stream(self.device).wait_stream(self.runner.post_stream)
            sums = torch.cat(self.runner.sums, dim=0) if len(self.runner.sums) > 1 else self.runner.sums[0]
        if write_event_frames:
            ub = _ef.upper_bound(sums, self.percentile, self.ceil, self.keep)
            frames = _ef.normalize(sums, ub, self.keep).cpu().numpy()
        return frames, ub, sums


@torch.no_grad()
def stream_clip(model, image_paths=None, vidcap=None, infer_type='center', seq_len=16, width=346, height=260,
                batch_size=1, fps=30, ceil=10, upper_bound_percentile=98, keep_polarity=True,
                write_event_frames=True, seed=0, pair_base=0, device=None, schedule=None, events_to_host=True,
                device_resize=None, keep_event_frame_sums=False, pano_fn=None):
    """Device-resident, pipelined version of v2ce.py:322-372 (runner.BatchRunner: the network of batch i+1 runs over
    the event frames + LDATI of batch i, results leave on a copy stream).  Returns ClipResult with the concatenated
    event stream (timestamps offset per frame, v2ce.py:365) and the uint8 BGR preview frames (clip-global percentile,
    as the reference computes it)."""
    assert image_paths is not None or vidcap is not None
    # pano_fn(model, image_units, width): replaces the serial tile loop of a pano batch (dist.py shares the tiles of a
    # window among ranks when a clip has fewer batches than ranks)
    pano = pano_fn if pano_fn is not None else _pano_device
    device = torch.device(device or 'cuda')
    frame_count = vidcap.frame_count if vidcap is not None else len(image_paths)
    # `schedule` = (window starts relative to this reader, mode): a rank's share of a longer clip (dist.py)
    starts, mode = schedule if schedule is not None else window_schedule(frame_count, seq_len)
    if len(starts) == 0:
        return ClipResult(np.empty(0, _ldati.EVENT_DTYPE), None, None, 0)
    # raw uint8 windows when the frames already have the model's height (the resize of image_pre_processing is then
    # the identity and the rest of it runs inside the head conv); float image units otherwise
    # (a clip of <= seq_len frames has a negative first start, v2ce.py:150-154: probe a frame that exists)
    probe = np.asarray(_read_window(image_paths, vidcap, max(int(starts[0]), 0), 0))
    # device_resize=False (or V2CE_DEVICE_RESIZE=0) keeps cv2.resize on the host, float units over PCIe
    if device_resize is None:
        device_resize = os.environ.get('V2CE_DEVICE_RESIZE', '1') not in ('', '0')
    route, infer = _frame_route(model, infer_type, probe.dtype, probe.shape, height, width, device_resize, pano)
    if route == 'native':
        batches = _window_batches_u8(image_paths, vidcap, seq_len, batch_size, schedule, width)
    elif route == 'raw':
        batches = _window_batches_u8(image_paths, vidcap, seq_len, batch_size, schedule, None)
    else:
        infer = (lambda u: _center_device(model, u, width)) if infer_type == 'center' else \
                (lambda u: pano(model, u, width))
        batches = _batches(image_paths, vidcap, seq_len, height, batch_size, schedule)
    plan = batch_plan(starts, mode, batch_size)
    _claim_model(model)
    try:
        with torch.cuda.device(device):
            clip = _ClipRun(model, device, infer, fps, ceil, upper_bound_percentile, keep_polarity, seed, pair_base,
                           keep_sums=write_event_frames or keep_event_frame_sums, hand_out=False,
                           clip_pairs=int(len(starts) * seq_len - ((seq_len - mode) if mode else 0)))
            runner = clip.runner
            prev = None
            for (x, _last), (_a, _e, trim) in zip(_background(batches), plan):
                t = clip.submit(x if x.is_pinned() else x.pin_memory(), trim)
                if prev is not None:
                    runner.wait(prev)                 # status check; the events stay on the device until the end
                prev = t
            if prev is not None:
                runner.wait(prev)
            events_dev, stream = runner.collected_events(to_host=events_to_host)   # False: ClipResult.event_stream is None
            frames, ub, sums = clip.event_frames(write_event_frames)
    finally:
        _release_model(model)
    res = ClipResult(stream, frames, ub, clip.pair_idx - pair_base)
    res.ef_sums_dev = sums if keep_event_frame_sums else None   # a sharded clip takes its percentile over all ranks (dist.py)
    res.event_stream_dev = events_dev            # the same bytes on the device (dist.py gathers from here)
    res.n_events = 0 if events_dev is None else events_dev.numel() // 13
    return res


def build_parser():
    """The reference's flags, verbatim (v2ce.py:283-302)."""
    parser = argparse.ArgumentParser()
    parser.add_argument('--fps', type=int, default=30, help='FPS of the output video')
    parser.add_argument('--seq_len', type=int, default=16, help='Sequence length')
    parser.add_argument('--ceil', type=int, default=10, help='The ceiling of the ef value')
    parser.add_argument('-u', '--upper_bound_percentile', type=int, default=98,
                        help='The percentile of the event frame nonzero values to set the upper bound during video writing')
    parser.add_argument('-f', '--image_folder', type=str, help='The folder containing the images to infer')
    parser.add_argument('-i', '--input_video_path', type=str, help='The path to the input video')
    parser.add_argument('-o', '--out_folder', type=str, default='./output', help='The folder to save the output video')
    parser.add_argument('-t', '--infer_type', type=str, default='center', help='The type of inference, can be center or pano')
    parser.add_argument('-m', '--model_path', type=str, default='./weights/v2ce_3d.pt', help='The path to the trained model')
    parser.add_argument('--out_name_suffix', type=str, default='', help='The suffix of the output video name')
    parser.add_argument('--max_frame_num', type=int, default=1800, help='The maximum number of frames to process')
    parser.add_argument('--width', type=int, default=346, help='The width of the frame/tensor input to the model')
    parser.add_argument('--height', type=int, default=260, help='The height of the frame/tensor input to the model')
    parser.add_argument('--write_event_frame_video', type=SBool, default=True, nargs='?', const=True,
                        help='Whether to write the event frame video')
    parser.add_argument('--vis_keep_polarity', type=SBool, default=True, nargs='?', const=True,
                        help='Whether to keep the polarity of the event frame during visualization')
    parser.add_argument('-l', '--log_level', type=str, default='info', help='Logging level')
    parser.add_argument('-b', '--batch_size', type=int, default=1, help='Batch size for inference')
    parser.add_argument('--stage2_batch_size', type=int, default=24, help='Batch size for inference')
    parser.add_argument('--seed', type=int, default=None,
                        help='(B200 extension) Philox key of the LDATI uniform draws; default: drawn from torch\'s RNG')
    return parser


def main(argv=None):
    import cv2
    args = build_parser().parse_args(argv)
    logging.basicConfig(level=getattr(logging, args.log_level.upper()))
    assert args.image_folder is not None or args.input_video_path is not None
    assert not (args.image_folder is not None and args.input_video_path is not None)
    if args.image_folder is not None:
        assert os.path.exists(args.image_folder), f'{args.image_folder} does not exist'
    if args.input_video_path is not None:
        assert os.path.exists(args.input_video_path), f'{args.input_video_path} does not exist'
    name = Path(args.image_folder).name if args.image_folder is not None else Path(args.input_video_path).stem
    output_name = f'{name}-ceil_{args.ceil}-fps_{args.fps}' if args.out_name_suffix == '' \
        else f'{name}-ceil_{args.ceil}-fps_{args.fps}-{args.out_name_suffix}'
    os.makedirs(args.out_folder, exist_ok=True)

    model = get_trained_mode(model_path=args.model_path)
    image_paths, vidcap = None, None
    if args.image_folder is not None:
        image_paths = sorted([op.join(args.image_folder, f) for f in os.listdir(args.image_folder)
                              if f.endswith('.png')])[:args.max_frame_num]
        logger.info(f'Now processing {args.image_folder}, Found {len(image_paths)} images.')
    else:
        from .scripts.video_reader import VideoReader
        vidcap = VideoReader(args.input_video_path, color_mode='GRAY')
        if args.max_frame_num is not None and 0 < args.max_frame_num < vidcap.frame_count:
            vidcap.frame_count = args.max_frame_num
        logger.info(f'Now processing {args.input_video_path}, processing {vidcap.frame_count} frames.')
    seed = args.seed if args.seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
    import time
    timings = {}
    t_start = time.perf_counter()
    res = stream_clip(model, image_paths=image_paths, vidcap=vidcap, infer_type=args.infer_type, seq_len=args.seq_len,
                      width=args.width, height=args.height, batch_size=args.batch_size, fps=args.fps, ceil=args.ceil,
                      upper_bound_percentile=args.upper_bound_percentile, keep_polarity=args.vis_keep_polarity,
                      write_event_frames=args.write_event_frame_video, seed=seed)
    timings['stream_clip_s'] = time.perf_counter() - t_start
    logger.info(f'Predicted voxel shape: ({res.n_pairs}, 2, 10, ...) (kept on the device)')
    encoder, encoder_error = None, []
    if args.write_event_frame_video:
        vis_color = 'rgb' if args.vis_keep_polarity else 'gray'
        ef_video_path = op.join(args.out_folder, f'{args.infer_type}-{output_name}-pred_ef_{vis_color}.mp4')
        logger.info(f'Upper bound of the event frame value during video writing: {res.ef_upper_bound}')

        def encode():                                 # v2ce.py:272-279; cv2 releases the GIL, so the mp4v encode
            try:                                      # runs beside the .npz write below (SURVEY.md N3)
                t_enc = time.perf_counter()
                H, W = res.ef_frames.shape[1:3]
                video = cv2.VideoWriter(ef_video_path, cv2.VideoWriter_fourcc(*'mp4v'), args.fps, (W, H))
                for f in res.ef_frames:
                    video.write(f)
                video.release()
                timings['encode_mp4v_s'] = time.perf_counter() - t_enc
            except Exception as e:                    # re-raised on the main thread
                encoder_error.append(e)

        import threading
        encoder = threading.Thread(target=encode, name='v2ce-ef-encode')
        encoder.start()
    logger.info(f'Generated event stream shape: , {res.event_stream.shape}')
    from .sink import save_npz
    t_npz = time.perf_counter()
    save_npz(op.join(args.out_folder, f'{output_name}-events.npz'), event_stream=res.event_stream)   # v2ce.py:371-372
    timings['save_npz_s'] = time.perf_counter() - t_npz
    if encoder is not None:
        encoder.join()
        if encoder_error:
            raise encoder_error[0]
        logger.info(f'Event frame video written to {ef_video_path}')
    timings['total_s'] = time.perf_counter() - t_start
    res.timings = timings
    logger.debug(f'stage times: {timings}')
    return res


if __name__ == '__main__':
    main()
