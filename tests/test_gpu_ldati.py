"""GPU parity: CUDA LDATI (through the C ABI) vs the CPU oracle and the reference goldens."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import ldati_oracle as lo, synth

pytestmark = pytest.mark.gpu


def _run(vox, **kw):
    from v2ce_toolbox_b200.scripts.LDATI import sample_voxel_statistical
    return sample_voxel_statistical(torch.as_tensor(vox).cuda(), **kw)


def _assert_rows_equal(got, want, what):
    assert len(got) == len(want), f'{what}: {len(got)} events vs {len(want)}'
    for f in ('timestamp', 'x', 'y', 'polarity'):
        assert np.array_equal(np.asarray(got[f]), np.asarray(want[f])), f'{what}: field {f} differs'


@pytest.mark.parametrize('bidirectional', [False, True])
def test_relocate_counts_bit_exact(bidirectional):
    """y_relocate alone (LDATI.py:80-123), both directions: counts and float32 tendencies bit for bit."""
    from v2ce_toolbox_b200 import _lib
    lib = _lib.load()
    relocate = lo.relocate_counts_bidirectional if bidirectional else lo.relocate_counts
    for (F, H, W) in ((3, 40, 52), (2, 33, 47), (1, 260, 346)):
        v = synth.make_voxels('mixed', F, H, W, seed=11)
        n, tend = relocate(v)
        vd = torch.from_numpy(v).cuda()
        cd = torch.empty((F, 2, 9, H, W), dtype=torch.int32, device='cuda')
        td = torch.empty((F, 2, 9, H, W), dtype=torch.float32, device='cuda')
        _lib.check(lib.v2ce_ldati_relocate(_lib.ptr(vd), F, H, W, int(bidirectional), _lib.ptr(cd), _lib.ptr(td),
                                           _lib.stream_ptr()))
        assert np.array_equal(cd.cpu().numpy(), n.astype(np.int32))
        assert np.array_equal(td.cpu().numpy().view(np.uint32), tend.view(np.uint32))


@pytest.mark.parametrize('kind,F,H,W', [('rand', 3, 40, 52), ('randint', 2, 24, 30), ('sparse', 3, 40, 52),
                                        ('mixed', 2, 33, 47), ('mixed', 2, 64, 80), ('rand', 1, 260, 346),
                                        ('randint', 1, 260, 346), ('sparse', 2, 260, 346)])
def test_events_bit_exact_vs_oracle(kind, F, H, W):
    v = synth.make_voxels(kind, F, H, W, seed=21)
    got = _run(v, fps=30, seed=1234, frame_base=7)
    want = lo.sample_voxel_statistical_oracle(v, fps=30, seed=1234, frame_base=7, flavor='cuda')
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.dtype.itemsize == 13
        _assert_rows_equal(g, w, f'{kind} frame {i}')


@pytest.mark.parametrize('fps', [24, 25, 60, 120, 1000])
def test_other_frame_rates(fps):
    v = synth.make_voxels('mixed', 2, 31, 45, seed=fps)
    got = _run(v, fps=fps, seed=5)
    want = lo.sample_voxel_statistical_oracle(v, fps=fps, seed=5, flavor='cuda')
    for i, (g, w) in enumerate(zip(got, want)):
        _assert_rows_equal(g, w, f'fps {fps} frame {i}')


def test_wide_elements_large_plane():
    # H*W needs 21 bits -> 64-bit sort elements
    v = synth.make_voxels('sparse', 1, 1080, 1920, seed=2) * np.float32(20)
    got = _run(v, fps=30, seed=3)
    want = lo.sample_voxel_statistical_oracle(v, fps=30, seed=3, flavor='cuda')
    _assert_rows_equal(got[0], want[0], 'wide')


def test_injected_draws_dense_tensor():
    from oracle import philox
    v = synth.make_voxels('randint', 2, 20, 28, seed=4)
    n, _ = lo.relocate_counts(v)
    M = int(n.max())
    d = philox.dense_draws(3, 2, 20, 28, M, seed=99)
    got = _run(v, fps=30, draws=torch.from_numpy(d).cuda())
    want = lo.sample_voxel_statistical_oracle(v, fps=30, draws=d, flavor='cuda')
    for i, (g, w) in enumerate(zip(got, want)):
        _assert_rows_equal(g, w, f'injected frame {i}')
    # the Philox stream evaluated in-kernel is the same function
    got2 = _run(v, fps=30, seed=99, frame_base=3)
    for g, g2 in zip(got, got2):
        _assert_rows_equal(g, g2, 'philox vs dense')


@pytest.mark.parametrize('name', ['kat', 'rand', 'randint', 'sparse', 'mixed24', 'mixed120'])
def test_cpu_flavour_against_reference_goldens(name, golden, golden_meta):
    """Kernel in torch-CPU scalar semantics vs the events the unmodified reference produced on CPU.
    Identical except where torch-CPU's non-IEEE float32 sqrt shifts a slope-sampled timestamp by 1 us
    (SURVEY.md F6): counts must match exactly, timestamps within 1 us on at most 1e-3 of the events;
    frames without multi-event pixels must match bit for bit."""
    g = golden('ldati')
    m = golden_meta['ldati'][name]
    v = g[f'{name}_voxel']
    got = _run(v, fps=m['fps'], seed=m['seed'], frame_base=m['frame_base'], flavor='cpu')
    n, _ = lo.relocate_counts(v)
    for i, ev in enumerate(got):
        ref = g[f'{name}_events_{i}'].view(lo.EVENT_DTYPE)
        assert len(ev) == len(ref)
        if n[i].max() <= 1:
            assert np.array_equal(lo.canonicalize(ev), ref)
        else:
            a, b = np.sort(ev['timestamp']), np.sort(ref['timestamp'])
            d = np.abs(a - b)
            assert d.max() <= 1 and (d != 0).mean() <= 1e-3


def test_full_size_digest_matches_reference_sparse(golden_meta):
    """346x260 sparse frame (single events only -> no sqrt): CUDA output hashes to the digest of the
    reference's own CPU output."""
    m = golden_meta['ldati']['full_sparse']
    v = synth.make_voxels('sparse', 1, 260, 346, seed=m['voxel_seed'])
    got = _run(v, fps=m['fps'], seed=m['seed'], frame_base=m['frame_base'], flavor='cpu')
    assert [len(g) for g in got] == m['counts']
    c = np.ascontiguousarray(lo.canonicalize(got[0]))
    assert hashlib.sha256(c.tobytes()).hexdigest() == m['sha256'][0]


def test_rejects_cpu_tensor_and_unsupported_modes():
    from v2ce_toolbox_b200 import V2ceError
    from v2ce_toolbox_b200.scripts.LDATI import sample_voxel_statistical
    with pytest.raises(V2ceError):
        sample_voxel_statistical(torch.zeros(1, 2, 10, 4, 4))
    with pytest.raises(AssertionError):                      # the reference's own assert (LDATI.py:135)
        sample_voxel_statistical(torch.zeros(1, 2, 10, 4, 4, device='cuda'), pooling_type='max')
    with pytest.raises(AssertionError):                      # the reference's own assert (LDATI.py:136)
        sample_voxel_statistical(torch.zeros(1, 2, 10, 4, 4, device='cuda'), additional_events_strategy='other')


OPTIONS = [(s_, b_) for s_ in ('slope', 'random', 'none') for b_ in (False, True) if (s_, b_) != ('slope', False)]


@pytest.mark.parametrize('strategy,bidirectional', OPTIONS)
@pytest.mark.parametrize('kind,F,H,W,fps', [('mixed', 2, 33, 47, 30), ('randint', 2, 24, 30, 24), ('rand', 2, 40, 52, 120),
                                            ('mixed', 1, 260, 346, 30)])
def test_options_bit_exact_vs_oracle(strategy, bidirectional, kind, F, H, W, fps):
    """SURVEY.md 8f N4: additional_events_strategy 'random' / 'none' and bidirectional=True through the same
    kernels, bit-exact against the oracle (torch-CUDA flavour), V=1 and V=4 pixel paths, full-size plane."""
    v = synth.make_voxels(kind, F, H, W, seed=31)
    kw = dict(fps=fps, seed=77, frame_base=3, additional_events_strategy=strategy, bidirectional=bidirectional)
    got = _run(v, **kw)
    want = lo.sample_voxel_statistical_oracle(v, flavor='cuda', **kw)
    for i, (g, w) in enumerate(zip(got, want)):
        _assert_rows_equal(g, w, f'{kind} {strategy} bidirectional={bidirectional} frame {i}')


@pytest.mark.parametrize('name', [f"{inp}-{s_}-{'bi' if b_ else 'uni'}" for inp in ('mixed24', 'randint')
                                  for (s_, b_) in OPTIONS])
def test_options_cpu_flavour_against_reference_goldens(name, golden, golden_meta):
    """Kernel in torch-CPU scalar semantics vs the unmodified reference's events for the off-CLI options.
    'random' and 'none' involve no sqrt, so they must match bit for bit (modulo the reference's undefined tie
    order); 'slope' is held to the criterion of test_cpu_flavour_against_reference_goldens."""
    m = golden_meta['ldati_options'][name]
    v = golden('ldati')[f"{m['input']}_voxel"]
    got = _run(v, fps=m['fps'], seed=m['seed'], frame_base=m['frame_base'], flavor='cpu',
               additional_events_strategy=m['additional_events_strategy'], bidirectional=m['bidirectional'])
    assert [len(e) for e in got] == m['counts']
    for i, ev in enumerate(got):
        ref = golden('ldati_options')[f'{name}_events_{i}'].view(lo.EVENT_DTYPE)
        if m['additional_events_strategy'] != 'slope':
            assert np.array_equal(lo.canonicalize(ev), ref), f'{name} frame {i}'
        else:
            d = np.abs(np.sort(ev['timestamp']) - np.sort(ref['timestamp']))
            assert d.max() <= 1 and (d != 0).mean() <= 1e-3


@pytest.mark.parametrize('kind,F,H,W,opts', [
    ('randint', 2, 24, 30, {}), ('mixed', 2, 33, 47, {}), ('rand', 1, 260, 346, {}), ('randint', 1, 260, 346, {}),
    ('mixed', 2, 40, 52, dict(additional_events_strategy='random')), ('mixed', 2, 33, 47, dict(bidirectional=True)),
    ('sparse', 3, 40, 52, dict(additional_events_strategy='none'))])
def test_emit_sort_and_pack_bit_exact(kind, F, H, W, opts):
    """Emit pass (per-warp totals handed over by the count pass), one-sweep sort and record writer produce the same
    bytes as the oracle: dense, sparse and mixed counts, V=1 and V=4 pixel paths, 32- and 64-bit elements, 2- and
    3-pass sorts, both relocation directions."""
    v = synth.make_voxels(kind, F, H, W, seed=51)
    want = lo.sample_voxel_statistical_oracle(v, fps=30, seed=9, frame_base=2, flavor='cuda', **opts)
    got = _run(v, fps=30, seed=9, frame_base=2, **opts)
    for j, (g, w) in enumerate(zip(got, want)):
        _assert_rows_equal(g, w, f'{kind} {opts} frame {j}')


def test_bidirectional_tendency_beyond_sort_window_raises():
    """bidirectional: bin 8's tendency is the tenth voxel bin itself (LDATI.py:108,111).  The sort-key window covers
    tendencies up to ldati.BIDIR_MAX_TENDENCY bins (rounded up to a power of two of microseconds, so < 2x that);
    a timestamp beyond it must fail loudly, never clamp silently."""
    from v2ce_toolbox_b200 import V2ceError, ldati
    v = np.zeros((1, 2, 10, 8, 12), np.float32)
    # one SINGLE event in bin 8 (floor(y8 + y9) == 1) whose tendency y9 is 4x outside the window; this needs a
    # negative voxel -- with the model's non-negative output a single event's tendency stays below 2 bins
    v[0, 0, 8, 3, 5] = -(4 * ldati.BIDIR_MAX_TENDENCY + 99.25)
    v[0, 0, 9, 3, 5] = 4 * ldati.BIDIR_MAX_TENDENCY + 100.5
    assert lo.relocate_counts_bidirectional(v)[0][0, 0, 8, 3, 5] == 1
    with pytest.raises(V2ceError):
        _run(v, bidirectional=True)
    v[0, 0, 8, 3, 5], v[0, 0, 9, 3, 5] = -2.0, 3.25          # tendency 3.25 bins: inside the window
    got = _run(v, bidirectional=True, seed=1)
    want = lo.sample_voxel_statistical_oracle(v, bidirectional=True, seed=1, flavor='cuda')
    assert want[0]['timestamp'].max() > int(1e6 / 30)                          # lands beyond the frame's end
    _assert_rows_equal(got[0], want[0], 'bidirectional tendency 3.25')


def test_empty_and_negative_inputs():
    v = np.zeros((2, 2, 10, 8, 12), np.float32)
    got = _run(v)
    assert [len(g) for g in got] == [0, 0]
    v = -np.abs(synth.make_voxels('rand', 1, 8, 12, seed=1))
    got = _run(v, seed=2)
    want = lo.sample_voxel_statistical_oracle(v, seed=2, flavor='cuda')
    _assert_rows_equal(got[0], want[0], 'negative')


@pytest.mark.parametrize('shift', [0, 1, 4, 13])
def test_output_buffer_of_any_alignment(shift):
    """v2ce_ldati_emit takes a caller pointer: the record writer uses 16-byte stores when the buffer allows it and word
    or byte stores otherwise; the bytes are the same."""
    from v2ce_toolbox_b200 import ldati
    v = synth.make_voxels('mixed', 2, 33, 47, seed=5)
    want = np.concatenate(lo.sample_voxel_statistical_oracle(v, fps=30, seed=3, flavor='cuda')).view(np.uint8)
    eng = ldati.LdatiEngine('cuda')
    vox = torch.from_numpy(v).cuda()
    params = ldati.make_params(2, 33, 47, fps=30, seed=3, device='cuda')
    seg = eng.count(vox, params)
    total = int(seg.sum())
    buf = torch.full((total * 13 + 64,), 0xAB, dtype=torch.uint8, device='cuda')
    out, status = eng.emit(vox, params, total, out=buf[shift:])
    got = buf.cpu().numpy()
    assert np.array_equal(got[shift:shift + total * 13], want)
    assert (got[:shift] == 0xAB).all() and (got[shift + total * 13:] == 0xAB).all()      # nothing outside the records
