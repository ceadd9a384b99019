"""LDATI, the event-frame preview and runner.BatchRunner at the sizes the product runs them, against the CPU oracle.

The bit-exact tests of tests/test_gpu_ldati*.py use at most three frame pairs per call.  The product sends 64 pairs per
call (BatchRunner: 4 windows x 16) and bench.py's LDATI record 100; there thousands of sort tiles chain their look-back
across hundreds of (frame, bin) segments, and byte offsets pass 2^31 and 2^32.  Checking every event of such a call with
the oracle would take minutes of CPU per row, so the tests rest on frame-split invariance (DESIGN.md §2):

  * every Philox draw is keyed by the global frame frame_base + f, never by the frame's place in the call, so frame f of an
    F-frame call must be byte-identical to a one-frame call on vox[f:f+1] with frame_base + f.  That is compared on the
    device for every frame of every row;
  * the per-(frame, bin) segment counts of every frame are compared with the oracle's relocation;
  * up to three frames per row (first, last, densest) are compared with the oracle bit for bit.

A second matrix pins the sort geometry (csrc/ldati.cu, make_geometry) at low frame rates and at the plane sizes where the
pixel field grows: each row checks every frame with the oracle and asserts the geometry property it exists for (element
width, key bit 31 in use, pass count), so a later change of the geometry cannot quietly make it redundant."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import baseline_oracle as bo, ef_oracle, ldati_oracle as lo, pipeline_oracle, synth

gpu = pytest.mark.gpu
H, W = 260, 346
SEED = 1234
FB = 1000                                   # frame_base of the big calls: a batch in the middle of a clip
LIMIT = (1 << 31) - (1 << 20)               # v2ce_ldati_emit refuses this many events or more (32-bit indices inside)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _geometry(params):
    """pix_bits, key_bits, element bytes and one-sweep pass count exactly as make_geometry / osw_passes in csrc/ldati.cu
    derive them from the parameters."""
    pix_bits = max(1, (params.height * params.width - 1).bit_length())     # least p >= 1 with 2^p >= H*W
    key_bits = max(1, int(params.key_span).bit_length())                   # least k >= 1 with 2^k >= key_span + 1
    elem = 8 if pix_bits + 1 + key_bits > 32 else 4
    return pix_bits, key_bits, elem, (key_bits + 5) // 6


def _emit_ws_bytes(params, total):
    from v2ce_toolbox_b200 import _lib
    n = ctypes.c_size_t()
    _lib.check(_lib.load().v2ce_ldati_emit_workspace_bytes(ctypes.byref(params), total, ctypes.byref(n)))
    return n.value


def _ws_bytes_per_element(params):
    """Sort-workspace growth per event: two element buffers plus < 2 bytes of per-tile tables."""
    n0, n1 = 1 << 23, 1 << 24
    return (_emit_ws_bytes(params, n1) - _emit_ws_bytes(params, n0)) / (n1 - n0)


def _ldati_call(eng, vox, frame_base, fps=30, **opts):
    """count -> emit into a fresh buffer; returns (records uint8 on the device, seg counts (F,9) host)."""
    from v2ce_toolbox_b200 import ldati
    F, _, _, h, w = vox.shape
    p = ldati.make_params(F, h, w, fps=fps, seed=SEED, frame_base=frame_base, device='cuda', **opts)
    seg = eng.count(vox, p).cpu().numpy()
    total = int(seg.sum())
    out, status = eng.emit(vox, p, total)
    ldati.check_status(status.cpu().numpy())
    return out[:total * 13], seg


def _baseline_call(vox, frame_base, mode):
    """The C-ABI calls of sample_methods.random_even_sample, with the records left on the device."""
    from v2ce_toolbox_b200 import _lib
    from v2ce_toolbox_b200._lib import check, ptr, stream_ptr
    from v2ce_toolbox_b200.sample_methods import random_even_sample as res
    lib = _lib.load()
    F, _, _, h, w = vox.shape
    p = res.make_params(F, h, w, fps=30, mode=mode, seed=SEED, frame_base=frame_base, device='cuda')
    n = ctypes.c_size_t()
    check(lib.v2ce_baseline_count_workspace_bytes(ctypes.byref(p), ctypes.byref(n)))
    cws = torch.empty(n.value, dtype=torch.uint8, device='cuda')
    counts = torch.empty(F, dtype=torch.int64, device='cuda')
    check(lib.v2ce_baseline_count(ptr(vox), ctypes.byref(p), ptr(cws), cws.numel(), ptr(counts), stream_ptr()))
    counts = counts.cpu().numpy()
    total = int(counts.sum())
    check(lib.v2ce_baseline_emit_workspace_bytes(ctypes.byref(p), total, ctypes.byref(n)))
    ews = torch.empty(n.value, dtype=torch.uint8, device='cuda')
    out = torch.empty(max(total, 1) * 13, dtype=torch.uint8, device='cuda')
    status = torch.zeros(4, dtype=torch.int32, device='cuda')
    check(lib.v2ce_baseline_emit(ptr(vox), ctypes.byref(p), ptr(cws), ptr(ews), ews.numel(), None, total, ptr(out),
                                 ptr(status), stream_ptr()))
    assert int(status.cpu()[0]) == 0
    return out[:total * 13], counts[:, None]


def _frame_starts(seg):
    """Byte offset of every frame's records in a call's output (seg: per-frame counts, (F, segments))."""
    return np.concatenate([[0], np.cumsum(seg.reshape(len(seg), -1).sum(axis=1))]) * 13


def _split_invariance(call, vox_dev, frame_base):
    """One F-frame call, then F one-frame calls: equal segment counts and equal bytes, frame by frame, on the device."""
    big, seg = call(vox_dev, frame_base)
    starts = _frame_starts(seg)
    for f in range(vox_dev.shape[0]):
        one, seg1 = call(vox_dev[f:f + 1], frame_base + f)
        assert np.array_equal(seg1[0], seg[f]), f'frame {f}: segment counts of the one-frame call differ'
        assert torch.equal(one, big[starts[f]:starts[f + 1]]), f'frame {f}: records differ from the one-frame call'
    return big, seg, starts


def _want_seg_counts(v, bidirectional=False):
    """The oracle's events per (frame, bin): every pixel-bin with n >= 1 relocated events emits n of them."""
    relocate = lo.relocate_counts_bidirectional if bidirectional else lo.relocate_counts
    step = max(1, (8 * H * W) // (v.shape[3] * v.shape[4]))             # bounds the host memory of the relocation
    return np.concatenate([np.clip(relocate(v[i:i + step])[0], 0, None).sum(axis=(1, 3, 4))
                           for i in range(0, len(v), step)])


def _sampled(seg, at_most=3):
    per_frame = seg.reshape(len(seg), -1).sum(axis=1)
    return sorted({0, len(seg) - 1, int(np.argmax(per_frame))})[:at_most]


def _assert_frame_bytes(big, starts, f, want, what):
    got = big[starts[f]:starts[f + 1]].cpu().numpy()
    want = np.ascontiguousarray(want).view(np.uint8).reshape(-1)
    assert got.size == want.size, f'{what} frame {f}: {got.size // 13} events vs {want.size // 13}'
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, f'{what} frame {f}: first differing event {bad[0] // 13}'


def _voxels(kind, F, h=H, w=W, seed=0):
    v = synth.make_voxels(kind, F, h, w, seed=seed)
    return v, torch.from_numpy(v).cuda()


# ---------------------------------------------------------------------------------------------------------------------
# 1. frame-split invariance at the product's call sizes
# ---------------------------------------------------------------------------------------------------------------------
SCALE_ROWS = [
    ('rand', 100, {}),                                                   # bench.py's LDATI chunk
    ('mixed', 64, {}),                                                   # BatchRunner's call
    ('sparse', 64, {}),                                                  # mostly empty segments
    ('randint', 72, {}),                                                 # element buffers > 2^31 B, records > 2^32 B
    ('mixed', 64, dict(additional_events_strategy='random')),            # 64-bit elements, 4 passes
    ('mixed', 64, dict(bidirectional=True)),
    ('mixed', 64, dict(additional_events_strategy='random', bidirectional=True)),
    ('mixed', 64, dict(pooling_type='avg', pooling_kernel_size=5)),      # pooled counts over many frames
]


@gpu
@pytest.mark.parametrize('kind,F,opts', SCALE_ROWS, ids=lambda x: x if isinstance(x, (str, int)) else
                         '-'.join(f'{k}={v}' for k, v in x.items()) or 'slope')
def test_ldati_frame_split_invariance_and_oracle(kind, F, opts):
    from v2ce_toolbox_b200 import ldati
    v, vd = _voxels(kind, F, seed=F)
    eng = ldati.LdatiEngine('cuda')
    big, seg, starts = _split_invariance(lambda x, fb: _ldati_call(eng, x, fb, **opts), vd, FB)
    assert np.array_equal(seg, _want_seg_counts(v, opts.get('bidirectional', False)))
    total = int(seg.sum())
    if kind == 'randint':
        assert total * 13 > 1 << 32 and total * 4 > 1 << 31 and total < LIMIT, total
        assert _geometry(ldati.make_params(F, H, W, flavor='cpu', device='cpu'))[2] == 4
    for f in _sampled(seg, 2 if kind == 'randint' else 3):
        want = lo.sample_voxel_statistical_oracle(v[f:f + 1], fps=30, seed=SEED, frame_base=FB + f, flavor='cuda', **opts)
        _assert_frame_bytes(big, starts, f, want[0], f'{kind} F={F} {opts}')


@gpu
def test_ldati_model_output_frame_split_invariance_and_oracle():
    """The distribution the product sees: 'reference'-init V2ce3d on synth.make_video, 4 windows x 16 pairs (bench.py)."""
    from v2ce_toolbox_b200 import ldati
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    from v2ce_toolbox_b200.v2ce import image_pre_processing
    frames = synth.make_video(65, H, W, seed=0)
    units = torch.stack([image_pre_processing(frames[s:s + 17], H) for s in (0, 16, 32, 48)], dim=0)
    m = V2ce3d()
    m.load_state_dict(synth.make_state_dict(0, 'reference'))
    m.eval().to('cuda')
    vd = m(units.cuda()).reshape(64, 2, 10, H, W).contiguous()
    del m
    v = vd.cpu().numpy()
    eng = ldati.LdatiEngine('cuda')
    big, seg, starts = _split_invariance(lambda x, fb: _ldati_call(eng, x, fb), vd, FB)
    assert np.array_equal(seg, _want_seg_counts(v))
    assert seg.sum() > 0
    for f in _sampled(seg):
        want = lo.sample_voxel_statistical_oracle(v[f:f + 1], fps=30, seed=SEED, frame_base=FB + f, flavor='cuda')
        _assert_frame_bytes(big, starts, f, want[0], 'model output')


@gpu
@pytest.mark.parametrize('mode', ['random', 'even'])
def test_baseline_frame_split_invariance_and_oracle(mode):
    """The baseline samplers sort whole frames (one segment per frame, 3 passes at 30 fps)."""
    v, vd = _voxels('mixed', 64, seed=3)
    big, seg, starts = _split_invariance(lambda x, fb: _baseline_call(x, fb, mode), vd, FB)
    for f in _sampled(seg):
        want = bo.sample_voxel_baseline_oracle(v[f:f + 1], fps=30, even=mode == 'even', random=mode == 'random',
                                               seed=SEED, frame_base=FB + f, flavor='cuda')
        _assert_frame_bytes(big, starts, f, want[0], f'baseline {mode}')


@gpu
def test_ldati_frame_split_invariance_wide_plane_over_4gib():
    """1080x1920 randint, 6 frames (~1.1 G events): 64-bit element buffers > 2^32 bytes.  An oracle frame would hold
    ~186 M events (over a minute of CPU each), so the oracle checks the counts of every frame; the events of this plane
    are held to the oracle by test_geometry_matrix_bit_exact's 1080x1920 row."""
    from v2ce_toolbox_b200 import ldati
    F, h, w = 6, 1080, 1920
    v, vd = _voxels('randint', F, h, w, seed=6)
    eng = ldati.LdatiEngine('cuda')
    p = ldati.make_params(F, h, w, fps=30, seed=SEED, frame_base=FB, device='cuda')
    seg = eng.count(vd, p).cpu().numpy()
    total = int(seg.sum())
    assert _geometry(p)[2] == 8 and total * 8 > 1 << 32 and total < LIMIT, total
    torch.cuda.empty_cache()
    need = int(1.25 * _emit_ws_bytes(p, total)) + 13 * total + 13 * int(seg.sum(axis=1).max()) + (1 << 30)
    free = torch.cuda.mem_get_info()[0]
    if free < need:
        pytest.skip(f'needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free')
    del seg
    _, seg, _ = _split_invariance(lambda x, fb: _ldati_call(eng, x, fb), vd, FB)
    assert np.array_equal(seg, _want_seg_counts(v))


# ---------------------------------------------------------------------------------------------------------------------
# 2. key- and pixel-width matrix, every frame against the oracle
# ---------------------------------------------------------------------------------------------------------------------
BIDI = dict(bidirectional=True)
RAND = dict(additional_events_strategy='random')
_OPT_NAMES = {'{}': 'slope', str(BIDI): 'bidirectional', str(RAND): 'random'}
# (kind, F, H, W, fps, opts, (key_bits, passes, element bytes), key reaches bit 31 of a 32-bit element)
GEOMETRY_ROWS = [
    ('mixed', 2, H, W, 1, {}, (17, 3, 8), False),
    ('mixed', 2, H, W, 1, RAND, (20, 4, 8), False),
    ('mixed', 2, H, W, 1, BIDI, (27, 5, 8), False),
    ('mixed', 2, H, W, 5, {}, (15, 3, 8), False),                        # 64-bit by one bit
    ('mixed', 2, H, W, 5, RAND, (20, 4, 8), False),
    ('mixed', 2, H, W, 5, BIDI, (25, 5, 8), False),
    ('mixed', 2, H, W, 10, {}, (14, 3, 4), True),
    ('mixed', 2, H, W, 10, RAND, (20, 4, 8), False),
    ('mixed', 2, H, W, 10, BIDI, (24, 4, 8), False),
    ('mixed', 2, H, W, 15, {}, (13, 3, 4), False),
    ('mixed', 2, H, W, 15, RAND, (20, 4, 8), False),
    ('mixed', 2, H, W, 15, BIDI, (23, 4, 8), False),
    ('mixed', 2, H, W, 23, {}, (13, 3, 4), False),
    ('mixed', 2, H, W, 23, RAND, (20, 4, 8), False),
    ('mixed', 2, H, W, 23, BIDI, (23, 4, 8), False),
    ('randint', 2, H, W, 10, {}, (14, 3, 4), True),                      # dense multi-event quads, key in bit 31
    ('mixed', 2, 512, 512, 30, {}, (12, 2, 4), False),                   # 2^18 pixels: 18-bit pixel field
    ('mixed', 2, 513, 512, 30, {}, (12, 2, 4), True),                    # just above: 19 bits, 32 bits in all
    ('rand', 1, 1080, 1920, 30, {}, (12, 2, 8), False),                  # 21-bit pixel field, ~20 M events
]


@gpu
@pytest.mark.parametrize('kind,F,h,w,fps,opts,geom,bit31', GEOMETRY_ROWS,
                         ids=[f"{r[0]}-{r[3]}x{r[2]}-fps{r[4]}-{_OPT_NAMES[str(r[5])]}" for r in GEOMETRY_ROWS])
def test_geometry_matrix_bit_exact(kind, F, h, w, fps, opts, geom, bit31):
    from v2ce_toolbox_b200 import ldati
    from v2ce_toolbox_b200.scripts.LDATI import sample_voxel_statistical
    p = ldati.make_params(F, h, w, fps=fps, device='cuda', **opts)
    pix_bits, key_bits, elem, passes = _geometry(p)
    assert (key_bits, passes, elem) == geom
    assert (elem == 4 and pix_bits + 1 + key_bits == 32) == bit31
    assert 2 * elem <= _ws_bytes_per_element(p) < 2 * elem + 2          # the library sizes the elements the same way
    v = synth.make_voxels(kind, F, h, w, seed=fps)
    kw = dict(fps=fps, seed=SEED, frame_base=FB, **opts)
    got = sample_voxel_statistical(torch.from_numpy(v).cuda(), **kw)
    want, seg = lo.sample_voxel_statistical_oracle(v, flavor='cuda', return_seg_counts=True, **kw)
    top = 0
    for f, (g, wf) in enumerate(zip(got, want)):
        assert len(g) == len(wf), f'frame {f}: {len(g)} events vs {len(wf)}'
        assert np.array_equal(np.ascontiguousarray(g).view(np.uint8), np.ascontiguousarray(wf).view(np.uint8)), \
            f'frame {f} differs'
        # largest sort key of the frame: ts - bin_base_us + KEY_BIAS per bin segment
        bins = np.repeat(np.arange(9), seg[f])
        keys = wf['timestamp'] - np.array(p.bin_base_us[:9], dtype=np.int64)[bins] + ldati.KEY_BIAS
        if keys.size:
            top = max(top, int(keys.max()))
    assert 0 < top < 1 << key_bits
    if bit31:
        assert top >= 1 << (key_bits - 1), 'no event sets bit 31 of its sort element'


# ---------------------------------------------------------------------------------------------------------------------
# 3. the per-call event limit
# ---------------------------------------------------------------------------------------------------------------------
def test_emit_workspace_query_at_the_event_limit():
    """Host only: the emit workspace query accepts 2^31 - 2^20 - 1 events and refuses 2^31 - 2^20."""
    from v2ce_toolbox_b200 import V2ceError, ldati
    for kw in (dict(), dict(bidirectional=True)):                        # 32- and 64-bit elements
        p = ldati.make_params(1, H, W, flavor='cpu', device='cpu', **kw)
        assert _emit_ws_bytes(p, LIMIT - 1) > 2 * 4 * (LIMIT - 1)
        with pytest.raises(V2ceError):
            _emit_ws_bytes(p, LIMIT)


@gpu
def test_call_over_the_event_limit_fails_before_allocating():
    """1080x1920 randint, 12 frames (~2.2 G events): the call raises V2ceError, and it does so before allocating the
    ~29 GB of records or the sort workspace: peak device allocation stays at voxels + count workspace."""
    from v2ce_toolbox_b200 import V2ceError, ldati
    from v2ce_toolbox_b200.scripts.LDATI import sample_voxel_statistical
    F, h, w = 12, 1080, 1920
    vox = torch.empty((F, 2, 10, h, w), dtype=torch.float32, device='cuda')
    vox.random_(0, 10, generator=torch.Generator(device='cuda').manual_seed(12))
    p = ldati.make_params(F, h, w, fps=30, seed=1, device='cuda')
    n = ctypes.c_size_t()
    from v2ce_toolbox_b200 import _lib
    _lib.check(_lib.load().v2ce_ldati_count_workspace_bytes(ctypes.byref(p), ctypes.byref(n)))
    total = int(ldati.LdatiEngine('cuda').count(vox, p).sum())
    assert total >= LIMIT, total
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with pytest.raises(V2ceError):
        sample_voxel_statistical(vox, fps=30, seed=1)
    peak = torch.cuda.max_memory_allocated() - base
    # a growing count workspace is allocated before the smaller one is freed
    assert peak <= 2.25 * n.value + (16 << 20), f'{peak} bytes allocated by a refused call (count workspace {n.value})'


# ---------------------------------------------------------------------------------------------------------------------
# 4. event-frame sums, select and normalise at scale
# ---------------------------------------------------------------------------------------------------------------------
EF_CASES = {'mixed-64x346x260': ('mixed', 64, H, W), 'pano-8x2076x1080': ('mixed', 8, 1080, 2076),
            'randint-64x346x260': ('randint', 64, H, W)}


def _integer_index_percentile(n):
    """A percentile q in (0, 100) for which numpy's virtual index (n - 1) * (q / 100) is exactly an integer."""
    for j in range((n - 1) // 3, n - 1):
        q = 100.0 * j / (n - 1)
        vi = (n - 1) * (q / 100.0)
        if vi == int(vi):
            return q
    raise AssertionError(n)


@gpu
@pytest.mark.parametrize('keep', [True, False], ids=['rgb', 'gray'])
@pytest.mark.parametrize('case', list(EF_CASES))
def test_event_frames_at_scale(case, keep):
    from v2ce_toolbox_b200 import event_frames as ef, ldati
    kind, N, h, w = EF_CASES[case]
    v = synth.make_voxels(kind, N, h, w, seed=N)
    if kind == 'mixed':
        v *= np.float32(0.3)                                            # percentiles below the ceiling
        v[0, :, :, :3] = 0                                              # exact zeros among the sums
    vd = torch.from_numpy(v).cuda()
    sums = ef.accumulate(vd, keep)
    want = ef_oracle.accumulate(v, keep)
    del v
    assert np.array_equal(sums.cpu().numpy().view(np.uint32), want.view(np.uint32))
    mult = 1 if keep else 3
    npos = int((want > 0).sum())
    no_ceil = float('inf')
    for q in (0, 2, 50, 98, 99.9, 100, _integer_index_percentile(npos * mult)):
        assert ef.upper_bound(sums, q, no_ceil, keep) == ef_oracle.upper_bound(want, q, no_ceil, keep), q
    # unaligned pointer, odd length: the select kernel's scalar path
    tail = sums.view(-1)[1:]
    assert tail.data_ptr() % 16 and tail.numel() % 4
    for q in (2, 50, 98):
        assert ef.upper_bound(tail, q, no_ceil, keep) == ef_oracle.upper_bound(want.reshape(-1)[1:], q, no_ceil, keep), q
    ub = ef_oracle.upper_bound(want, 98, 10, keep)
    assert ef.upper_bound(sums, 98, 10, keep) == ub
    assert np.array_equal(ef.normalize(sums, ub, keep).cpu().numpy(), ef_oracle.to_bgr_u8(want, ub, keep))
    if keep and h == H:
        # the LDATI count pass writes the same sums from its own read of the voxels (BatchRunner's route)
        fused = torch.full_like(sums, float('nan'))
        ldati.LdatiEngine('cuda').count(vd, ldati.make_params(N, h, w, fps=30, seed=1, device='cuda'), ef_sums=fused)
        assert torch.equal(fused, sums)


# ---------------------------------------------------------------------------------------------------------------------
# 5. BatchRunner at the benchmark's shape
# ---------------------------------------------------------------------------------------------------------------------
def _check_ticket(t, vox_dev, fps=30, seed=0, oracle_frames=2):
    """Ticket t of a BatchRunner against one plain LDATI call on the same voxels (frame_base = pair_base, plus the
    per-frame timestamp offsets), sampled oracle frames, and the event-frame oracle."""
    from v2ce_toolbox_b200 import ldati
    n = vox_dev.shape[0]
    p = ldati.make_params(n, H, W, fps=fps, seed=seed, frame_base=t.pair_base, device='cuda', add_frame_offset=True)
    eng = ldati.LdatiEngine('cuda')
    seg = eng.count(vox_dev, p).cpu().numpy()
    assert np.array_equal(t.seg_counts, seg)
    total = int(seg.sum())
    offs = torch.from_numpy(ldati.frame_offsets_us(t.pair_base, n, fps)).cuda()
    want, status = eng.emit(vox_dev, p, total, frame_offsets=offs)
    ldati.check_status(status.cpu().numpy())
    assert t.total == total and torch.equal(t.events_dev[:total * 13], want[:total * 13])
    del want
    v = vox_dev.cpu().numpy()
    starts = _frame_starts(seg)
    for f in sorted({0, n - 1})[:oracle_frames]:
        wf = lo.sample_voxel_statistical_oracle(v[f:f + 1], fps=fps, seed=seed, frame_base=t.pair_base + f,
                                                flavor='cuda')[0]
        wf['timestamp'] += pipeline_oracle.frame_offset_us(t.pair_base + f, fps)
        _assert_frame_bytes(t.events_dev, starts, f, wf, f'batch at pair {t.pair_base}')
    sums = ef_oracle.accumulate(v, True)
    ub = ef_oracle.upper_bound(sums, 98, 10, True)
    assert t.ub == ub
    assert np.array_equal(t.frames_dev.cpu().numpy(), ef_oracle.to_bgr_u8(sums, ub, True))


@gpu
def test_batch_runner_bench_shape_with_slot_reuse():
    """346x260, 4 windows x 16 pairs, three slots.  Densities change from batch to batch, so every slot is reused by a
    batch with more events than its previous user and by one with fewer (slot 0: sparse -> randint -> sparse, slot 1:
    randint -> sparse, slot 2: rand -> mixed); the last batch keeps 5 pairs of its last window (a clip's pulled-back
    window).  Each batch is collected after the next one is submitted, as bench.py does."""
    from v2ce_toolbox_b200.runner import BatchRunner
    kinds = ['sparse', 'randint', 'rand', 'randint', 'sparse', 'mixed', 'sparse']
    queue = []
    runner = BatchRunner(None, 'cuda', fps=30, seed=0, copy_out=False, infer=lambda x: queue.pop(0))
    token = torch.zeros(1, device='cuda')
    pending, pair_base = None, 0
    for i, kind in enumerate(kinds):
        vox = torch.from_numpy(synth.make_voxels(kind, 64, H, W, seed=90 + i)).cuda()
        trim = 5 if i == len(kinds) - 1 else 0
        queue.append(vox.view(4, 16, 20, H, W))
        t = runner.submit(token, pair_base, trim_last_window_to=trim)
        if trim:
            vox = torch.cat([vox[:48], vox[64 - trim:]]).contiguous()
        assert t.n_pairs == vox.shape[0]
        if pending is not None:
            runner.wait(pending[0])
            _check_ticket(*pending, oracle_frames=1 if kinds[i - 1] == 'randint' else 2)
        pending = (t, vox)
        pair_base += t.n_pairs
    runner.flush()
    runner.wait(pending[0])
    _check_ticket(*pending)


@gpu
def test_batch_runner_real_model_uint8_and_units_routes():
    """One bench batch through the real model: raw uint8 windows (pre-processing fused into the head conv) and
    host-preprocessed image units give the same events and frames, and both match LDATI and the oracles."""
    from v2ce_toolbox_b200.runner import BatchRunner
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    from v2ce_toolbox_b200.v2ce import image_pre_processing
    frames = synth.make_video(65, H, W, seed=0)
    windows = np.stack([frames[s:s + 17] for s in (0, 16, 32, 48)], axis=0)
    units = torch.stack([image_pre_processing(w_, H) for w_ in windows], dim=0)
    results = []
    for x in (torch.from_numpy(windows).pin_memory(), units.pin_memory()):
        m = V2ce3d()                                    # one model per route: the spectral-norm state advances per call
        m.load_state_dict(synth.make_state_dict(0, 'reference'))
        runner = BatchRunner(m.eval().to('cuda'), 'cuda', fps=30, seed=0, copy_out=True)
        runner.keep_vox = True
        t = runner.submit(x, pair_base=64)
        ev, fr = runner.wait(t)
        _check_ticket(t, t.vox)
        results.append((ev, fr, t.ub))
    (ev_a, fr_a, ub_a), (ev_b, fr_b, ub_b) = results
    assert len(ev_a) > 0 and ub_a == ub_b
    assert np.array_equal(ev_a.view(np.uint8), ev_b.view(np.uint8)) and np.array_equal(fr_a, fr_b)
