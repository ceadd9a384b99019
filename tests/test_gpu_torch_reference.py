"""End-to-end pin of the kernels' `cuda` flavour against torch-CUDA itself (SURVEY.md 8c: "primary parity oracle = the
reference run on the same B200 through torch-CUDA").  torch_reference.py issues the reference's torch operations
(/root/reference/scripts/LDATI.py:13-51,80-123,126-214,217-310) on device='cuda' -- so the reciprocal-multiply scalar
divisions, the float32 arange, the IEEE sqrt, cuDNN's conv1d/conv2d/AvgPool2d are the real ones, not the oracle's model
of them -- with the SAME injected uniform draws as v2ce_ldati_emit (SURVEY.md F7) and a stable argsort (F5).
Bit-exact on all four record fields, row by row.  (On CPU the same restatement is pinned to the unmodified
reference: tests/test_torch_reference.py.)"""
import numpy as np
import pytest
import torch

import torch_reference as tr

pytestmark = pytest.mark.gpu


def _vox(kind, B, H, W, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    if kind == 'rand':
        return torch.rand((B, 2, 10, H, W), generator=g, device='cuda')
    if kind == 'randint':
        return torch.randint(0, 10, (B, 2, 10, H, W), generator=g, device='cuda').float()
    if kind == 'sparse':
        return torch.rand((B, 2, 10, H, W), generator=g, device='cuda') * 0.015
    v = torch.rand((B, 2, 10, H, W), generator=g, device='cuda') * 3
    v[torch.rand(v.shape, generator=g, device='cuda') < 0.5] = 0
    return v


def _compare(vox, fps=30, **opts):
    from v2ce_toolbox_b200.scripts.LDATI import sample_voxel_statistical
    B, _, _, H, W = vox.shape
    g = torch.Generator(device='cuda').manual_seed(99)
    draws = torch.rand((B, 2, 9, H, W, 24), generator=g, device='cuda')
    want = tr.sample_voxel_statistical_torch(vox, fps=fps, draws=draws, stable=True, **opts)
    got = sample_voxel_statistical(vox, fps=fps, draws=draws, flavor='cuda', **opts)
    n = 0
    for a, b in zip(got, want):
        assert len(a) == len(b), (len(a), len(b))
        for f in ('timestamp', 'x', 'y', 'polarity'):
            assert np.array_equal(np.asarray(a[f]), np.asarray(b[f])), f
        n += len(a)
    return n


@pytest.mark.parametrize('kind', ['rand', 'randint', 'mixed', 'sparse'])
def test_kernels_equal_torch_cuda_at_346x260(kind):
    """The CLI's options (slope, no pooling, unidirectional) at the DAVIS346 resolution, two frames."""
    n = _compare(_vox(kind, 2, 260, 346, 42))
    assert n > 0


@pytest.mark.parametrize('opts', [dict(additional_events_strategy='random'), dict(additional_events_strategy='none'),
                                  dict(bidirectional=True), dict(pooling_type='weighted'),
                                  dict(pooling_type='avg', pooling_kernel_size=3),
                                  dict(bidirectional=True, pooling_type='avg', pooling_kernel_size=5)])
@pytest.mark.parametrize('kind', ['randint', 'mixed'])
def test_kernels_equal_torch_cuda_options(kind, opts):
    _compare(_vox(kind, 2, 37, 53, 7), **opts)


@pytest.mark.parametrize('fps', [1, 5, 10, 24, 60, 120, 1000])
def test_kernels_equal_torch_cuda_frame_rates(fps):
    _compare(_vox('mixed', 1, 64, 96, fps), fps=fps)


def test_unet_against_torch_cuda_fp32_and_tf32():
    """V2ce3d (bf16 operands, fp32 accumulation) against cuDNN's conv3d on the same device: true fp32
    (allow_tf32=False) is the reference value; the TF32 run shows what upstream's default CUDA path itself deviates by."""
    from oracle import synth
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    sd = synth.make_state_dict(0, 'reference')
    x = torch.randn(1, 16, 2, 260, 346, generator=torch.Generator().manual_seed(3)).cuda()
    ours = V2ce3d()
    ours.load_state_dict(sd)
    ours.eval().to('cuda')
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        ref32 = tr.TorchV2ce3d(sd, 'cuda')
        torch.backends.cudnn.allow_tf32 = True
        reftf = tr.TorchV2ce3d(sd, 'cuda')
        for call in range(2):                                # spectral-norm state advances with every call
            y = ours(x)
            torch.backends.cudnn.allow_tf32 = False
            r32 = ref32(x)
            torch.backends.cudnn.allow_tf32 = True
            rtf = reftf(x)
            rel = float((y - r32).norm() / r32.norm())
            mx = float((y - r32).abs().max() / r32.abs().max())
            rel_tf = float((rtf - r32).norm() / r32.norm())
            print(f'call {call}: ours vs cuDNN-fp32 rel-L2 {rel:.3e} max-abs/max {mx:.3e}; cuDNN-TF32 vs fp32 rel-L2 {rel_tf:.3e}')
            from conftest import record_measurement
            record_measurement('voxel_vs_cudnn_fp32', shape=[1, 16, 2, 260, 346], call=call, rel_l2=rel, max_abs_over_max=mx,
                               cudnn_tf32_rel_l2=rel_tf)
            assert rel <= 1e-2 and mx <= 3e-2, (rel, mx)     # SURVEY.md F10: the calibrated bf16 tolerance
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
