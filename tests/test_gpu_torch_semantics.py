"""Evidence for the 'cuda' arithmetic flavour of the LDATI oracle (SURVEY.md F6): each scalar
semantic the flavour assumes is checked against torch-CUDA itself on the B200.  These are the
torch ops the reference executes at scripts/LDATI.py:156,163-164,188,190,195-196,209-212."""
import numpy as np
import pytest
import torch

from oracle import ldati_oracle as lo

pytestmark = pytest.mark.gpu
F32 = np.float32


@pytest.mark.parametrize('fps', [1, 5, 10, 24, 25, 30, 50, 60, 120, 240, 1000])
def test_arange_bin_starts(fps):
    got = torch.arange(0, 1 / fps, 1 / fps / 9, device='cuda').cpu().numpy()
    assert got.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), lo.bin_starts(fps, 9, 'cuda').view(np.uint32))


def test_division_by_python_scalar_is_reciprocal_multiply():
    g = torch.Generator(device='cpu').manual_seed(0)
    x32 = torch.rand(1 << 16, generator=g)
    x64 = x32.double()
    for fps in (1, 5, 10, 24, 30, 120):
        k = lo.Consts(fps, 0, 'cuda')
        got = (x64.cuda() / fps / 9).cpu().numpy()
        assert np.array_equal(got, x64.numpy() * k.r_fps64 * k.r_c64)
        got = (x32.cuda() / fps / 9).cpu().numpy()
        assert np.array_equal(got, (x32.numpy() * k.r_fps32) * k.r_c32)
        vs2 = (1 / fps / 9) ** 2
        got = (x32.cuda() / vs2).cpu().numpy()
        assert np.array_equal(got, x32.numpy() * k.r_vs2_32)
    S = torch.arange(-30, 31, dtype=torch.float32)
    got = ((3 * S.cuda() - 0 * S.cuda()) / (3 * 2 - 0 ** 2)).cpu().numpy()
    assert np.array_equal(got, (F32(3) * S.numpy() - F32(0)) * F32(1.0 / 6))


def test_sqrt_and_tensor_division_are_ieee():
    g = torch.Generator(device='cpu').manual_seed(1)
    x = torch.rand(1 << 18, generator=g) * 3e5
    y = torch.rand(1 << 18, generator=g) * 7 + 0.1
    assert np.array_equal(torch.sqrt(x.cuda()).cpu().numpy(), np.sqrt(x.numpy()))
    assert np.array_equal((x.cuda() / y.cuda()).cpu().numpy(), x.numpy() / y.numpy())
    assert np.array_equal((x.cuda() ** 2).cpu().numpy(), x.numpy() * x.numpy())


def test_nan_to_long_on_cuda():
    # not what the PTX manual's "NaN converts to 0" suggests: torch-CUDA yields INT64_MIN, like x86
    t = torch.tensor([float('nan'), 1.9, -1.9], device='cuda').to(torch.long).cpu().numpy()
    assert t.tolist() == [np.iinfo(np.int64).min, 1, -1]


def test_slope_params_match_torch_cuda_ops():
    """k and b of LDATI.py:184-188 evaluated with torch-CUDA ops vs the oracle's cuda flavour."""
    rng = np.random.default_rng(0)
    n = rng.integers(0, 12, (4, 9, 16, 16)).astype(np.int64)
    k = lo.Consts(30, 0, 'cuda')
    kk, b = lo.slope_params(n, k)
    y = torch.from_numpy(n).cuda().float()
    S = torch.zeros_like(y)
    S[:, 1:-1] = y[:, 2:] - y[:, :-2]
    voxel_step = 1 / 30 / 9
    kt = ((3 * S - 0 * y) / (3 * 2 - 0 ** 2)) / (voxel_step ** 2) / (y + 1e-8)
    bt = 1 / voxel_step - voxel_step * kt / 2
    assert np.array_equal(kt.cpu().numpy().view(np.uint32), kk.view(np.uint32))
    assert np.array_equal(bt.cpu().numpy().view(np.uint32), b.view(np.uint32))


def test_pooled_slope_ops_are_float32_on_cuda():
    """pooling_type 'avg' / 'weighted' (LDATI.py:176-183 then :25-39): AvgPool2d / conv2d on the counts, then the
    [-1, 0, 1] conv1d over bins.  The oracle's cuda flavour takes all three as float32 arithmetic; cuDNN may instead
    run the convolutions on TF32 tensor cores (torch.backends.cudnn.allow_tf32 defaults to True), which is exact for
    'weighted' (dyadic weights, small integers) but not for the k/9-valued 'avg' counts."""
    import torch.nn.functional as Fn
    g = torch.Generator(device='cpu').manual_seed(5)
    n = torch.randint(0, 12, (4, 9, 20, 24), generator=g).float()
    n_np = n.numpy().astype(np.int64)
    avg = torch.nn.AvgPool2d(kernel_size=3, stride=1, padding=1)(n.cuda()).cpu().numpy()
    assert np.array_equal(avg.view(np.uint32), lo.pool_counts(n_np, 'avg', 3).view(np.uint32))
    kern = (torch.tensor([[1, 2, 1], [2, 4, 2], [1, 2, 1]], dtype=torch.float) / 16).reshape(1, 1, 3, 3).cuda()
    wgt = Fn.conv2d(n.reshape(36, 1, 20, 24).cuda(), kern, padding=1).reshape(4, 9, 20, 24).cpu().numpy()
    assert np.array_equal(wgt.view(np.uint32), lo.pool_counts(n_np, 'weighted').view(np.uint32))
    # the slope's conv1d on k/9-valued inputs: float32 subtraction of the two outer taps, or TF32-rounded inputs?
    yp = torch.from_numpy(avg)
    padded = Fn.pad(yp, (0, 0, 0, 0, 1, 1), mode='reflect')
    flat = torch.einsum('bkhw->bhwk', padded).reshape(4 * 20 * 24, 1, 11).cuda()
    xy = torch.tensor([-1.0, 0.0, 1.0], device='cuda').repeat(1, 1, 1)
    got = Fn.conv1d(flat, xy, padding=0).view(4, 20, 24, 9).permute(0, 3, 1, 2).cpu().numpy()
    want = np.zeros_like(avg)
    want[:, 1:-1] = avg[:, 2:] - avg[:, :-2]
    assert np.array_equal(got.view(np.uint32), want.astype(np.float32).view(np.uint32))
