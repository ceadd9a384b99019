"""GPU parity for stage 1: the tcgen05 implicit-GEMM conv (layer hook) against torch fp32 conv3d on
the same bf16-rounded operands, and the whole V2ce3d forward against the fp32 CPU oracle."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle.unet_oracle import UNetOracle
from conftest import record_measurement

pytestmark = pytest.mark.gpu


def conv_hook(src0, src1, hin, win, w, scale, shift, residual, act, ksize, stride, impl=0):
    """src0 (B,D,H0,W0,C0) bf16, src1 (B,D,Hin,Win,C1) bf16 | None -> out (B,D,Hout,Wout,Cout) bf16."""
    from v2ce_toolbox_b200 import _lib
    lib = _lib.load()
    B, D, H0, W0, C0 = src0.shape
    C1 = 0 if src1 is None else src1.shape[-1]
    cout = w.shape[0]
    pad = ksize // 2
    hout = (hin + 2 * pad - ksize) // stride + 1
    wout = (win + 2 * pad - ksize) // stride + 1
    out = torch.full((B, D, hout, wout, cout), float('nan'), dtype=torch.bfloat16, device='cuda')
    wh = np.ascontiguousarray(w.cpu().numpy(), dtype=np.float32)
    sh = np.ascontiguousarray(scale.cpu().numpy(), dtype=np.float32)
    th = np.ascontiguousarray(shift.cpu().numpy(), dtype=np.float32)
    _lib.check(lib.v2ce_conv3d_bf16_ex(_lib.ptr(src0), C0, H0, W0, _lib.ptr(src1), C1, B, D, hin, win, ksize, stride,
                                       wh.ctypes.data_as(ctypes.c_void_p), cout, sh.ctypes.data_as(ctypes.c_void_p),
                                       th.ctypes.data_as(ctypes.c_void_p), _lib.ptr(residual), act, _lib.ptr(out),
                                       impl, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return out


def torch_ref(src0, src1, hin, win, w, scale, shift, residual, act, ksize, stride):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    x = src0.float().permute(0, 4, 1, 2, 3)                       # (B,C,D,H,W)
    if src0.shape[2] != hin or src0.shape[3] != win:
        hi = (torch.arange(hin, device=x.device) * src0.shape[2]) // hin
        wi = (torch.arange(win, device=x.device) * src0.shape[3]) // win
        x = x[:, :, :, hi][:, :, :, :, wi]
    if src1 is not None:
        x = torch.cat([x, src1.float().permute(0, 4, 1, 2, 3)], dim=1)
    wq = w.to(torch.bfloat16).float()
    y = F.conv3d(x.double(), wq.double().cuda(), None, (1, stride, stride), ksize // 2).float()
    y = y * scale.cuda().view(1, -1, 1, 1, 1) + shift.cuda().view(1, -1, 1, 1, 1)
    y = y.permute(0, 2, 3, 4, 1)
    if residual is not None:
        y = y + residual.float()
    if act == 1:
        y = torch.relu(y)
    elif act == 2:
        y = F.leaky_relu(y, 0.01)
    return y


CASES = [
    # name, B, D, Hin, Win, C0, (H0,W0) or None, C1, Cout, k, stride, residual, act
    ('gemm32', 1, 2, 8, 16, 64, None, 0, 32, 1, 1, False, 0),
    ('gemm64', 1, 2, 8, 16, 64, None, 0, 64, 1, 1, False, 0),
    ('gemm128', 1, 2, 8, 16, 128, None, 0, 128, 1, 1, False, 1),
    ('gemm256', 1, 2, 8, 16, 64, None, 0, 256, 1, 1, False, 0),
    ('gemm512', 1, 2, 8, 16, 256, None, 0, 512, 1, 1, True, 1),
    ('k1_cin32', 1, 3, 9, 11, 32, None, 0, 64, 1, 1, False, 0),
    ('k3_s1', 1, 3, 9, 11, 64, None, 0, 64, 3, 1, False, 1),
    ('k3_s2_cin32', 2, 3, 9, 11, 32, None, 0, 64, 3, 2, False, 1),
    ('k1_s2', 1, 3, 9, 11, 64, None, 0, 128, 1, 2, False, 0),
    ('k3_res_relu', 1, 4, 10, 12, 128, None, 0, 128, 3, 1, True, 1),
    ('k3_leaky', 1, 2, 7, 9, 64, None, 0, 32, 3, 1, False, 2),
    ('concat_up_k3', 1, 3, 9, 11, 64, (5, 6), 32, 32, 3, 1, False, 1),
    ('concat_up_k1', 1, 3, 9, 11, 64, (5, 6), 32, 32, 1, 1, False, 0),
    ('concat_up_768', 1, 2, 9, 11, 512, (5, 6), 256, 256, 3, 1, False, 1),
    ('deepk_512', 1, 4, 6, 7, 512, None, 0, 512, 3, 1, True, 1),
    ('many_tiles', 2, 16, 33, 44, 64, None, 0, 64, 3, 1, True, 1),
]


# 3x3x3 stride-1 cases for the halo-tile kernel (channel pitches multiple of 64, no upsample)
HALO_CASES = [
    ('halo_64_64', 1, 3, 9, 11, 64, None, 0, 64, 3, 1, False, 1),
    ('halo_n32', 1, 3, 9, 11, 64, None, 0, 32, 3, 1, False, 0),
    ('halo_128_res', 1, 4, 10, 12, 128, None, 0, 128, 3, 1, True, 1),
    ('halo_two_src', 1, 3, 9, 11, 64, None, 64, 32, 3, 1, False, 2),
    ('halo_512', 1, 4, 6, 7, 512, None, 0, 512, 3, 1, True, 1),
    ('halo_768', 1, 2, 9, 11, 512, None, 256, 256, 3, 1, False, 1),
    ('halo_wide', 1, 2, 20, 70, 64, None, 0, 64, 3, 1, False, 1),
    ('halo_many', 2, 16, 33, 44, 64, None, 0, 64, 3, 1, True, 1),
    ('halo_fullres_slice', 1, 2, 260, 346, 64, None, 64, 32, 3, 1, False, 1),
]

# same, through the depth-merged variant (Cout <= 64, depth % 8 == 0): one and two depth blocks, two sources,
# two N tiles, residual, full-resolution tile shape
KDM_CASES = [
    ('kdm_n32', 1, 8, 9, 11, 64, None, 0, 32, 3, 1, False, 0),
    ('kdm_two_src_d16', 1, 16, 9, 11, 64, None, 64, 32, 3, 1, True, 1),
    ('kdm_n64_many', 2, 16, 33, 44, 64, None, 0, 64, 3, 1, True, 1),
    ('kdm_128_in', 1, 8, 20, 70, 128, None, 64, 64, 3, 1, False, 2),
    ('kdm_fullres', 1, 8, 260, 346, 64, None, 64, 32, 3, 1, True, 1),
    # stride (1,2,2) through the four parity views (one source): odd and even planes, 1-4 N tiles, 1-2 channel chunks
    ('kdm_s2_small', 1, 8, 9, 11, 64, None, 0, 32, 3, 2, False, 1),
    ('kdm_s2_odd', 2, 16, 33, 44, 64, None, 0, 64, 3, 2, False, 1),
    ('kdm_s2_128', 1, 8, 20, 70, 128, None, 0, 128, 3, 2, False, 2),
    ('kdm_s2_fullres', 1, 8, 260, 346, 64, None, 0, 64, 3, 2, False, 1),
]


@pytest.mark.parametrize('case', CASES + HALO_CASES + KDM_CASES, ids=[c[0] for c in CASES + HALO_CASES + KDM_CASES])
def test_conv_layer_vs_torch(case):
    name, B, D, hin, win, C0, up, C1, cout, k, stride, use_res, act = case
    impl = 2 if name.startswith('kdm') else 1 if name.startswith('halo') else 0
    g = torch.Generator(device='cpu').manual_seed(hash(name) % 1000)
    h0, w0 = up if up else (hin, win)
    src0 = torch.randn(B, D, h0, w0, C0, generator=g).to(torch.bfloat16).cuda()
    src1 = torch.randn(B, D, hin, win, C1, generator=g).to(torch.bfloat16).cuda() if C1 else None
    cin = C0 + C1
    w = torch.randn(cout, cin, k, k, k, generator=g) / np.sqrt(cin * k ** 3)
    scale = 0.5 + torch.rand(cout, generator=g)
    shift = 0.2 * torch.randn(cout, generator=g)
    pad = k // 2
    hout, wout = (hin + 2 * pad - k) // stride + 1, (win + 2 * pad - k) // stride + 1
    res = torch.randn(B, D, hout, wout, cout, generator=g).to(torch.bfloat16).cuda() if use_res else None
    out = conv_hook(src0, src1, hin, win, w, scale, shift, res, act, k, stride, impl=impl)
    ref = torch_ref(src0, src1, hin, win, w, scale, shift, res, act, k, stride)
    assert not torch.isnan(out.float()).any(), 'unwritten outputs'
    err = (out.float() - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 2e-3          # bf16 output rounding + fp32 accumulation-order noise
    bad = (err > tol).sum().item()
    assert bad == 0, f'{name}: {bad} of {err.numel()} outside tolerance, max err {err.max().item():.4g}'


@pytest.mark.parametrize('case', KDM_CASES, ids=[c[0] + '_shortcut' for c in KDM_CASES])
def test_conv_with_fused_shortcut_vs_torch(case):
    """Depth-merged kernel with the block's 1x1x1 shortcut conv fused in (impl 3 of the hook): both outputs."""
    name, B, D, hin, win, C0, up, C1, cout, k, stride, use_res, act = case
    g = torch.Generator(device='cpu').manual_seed(hash(name) % 1000 + 1)
    src0 = torch.randn(B, D, hin, win, C0, generator=g).to(torch.bfloat16).cuda()
    src1 = torch.randn(B, D, hin, win, C1, generator=g).to(torch.bfloat16).cuda() if C1 else None
    cin = C0 + C1
    w = torch.randn(cout, cin, 3, 3, 3, generator=g) / np.sqrt(cin * 27)
    w[:, :, 1, 1, 1] *= 4.0                      # the shortcut weights: make them count
    scale = 0.5 + torch.rand(cout, generator=g)
    shift = 0.2 * torch.randn(cout, generator=g)
    hout, wout = (hin - 1) // stride + 1, (win - 1) // stride + 1
    out2 = torch.full((B, D, hout, wout, cout), float('nan'), dtype=torch.bfloat16, device='cuda')
    out = conv_hook(src0, src1, hin, win, w, scale, shift, out2, act, 3, stride, impl=3)
    ref = torch_ref(src0, src1, hin, win, w, scale, shift, None, act, 3, stride)
    ref2 = torch_ref(src0, src1, hin, win, w[:, :, 1:2, 1:2, 1:2].contiguous(), scale, shift, None, 0, 1, stride)
    for got, want, what in ((out, ref, 'conv'), (out2, ref2, 'shortcut')):
        assert not torch.isnan(got.float()).any(), f'{what}: unwritten outputs'
        err = (got.float() - want).abs()
        tol = 2.0 ** -8 * want.abs() + 2e-3
        bad = (err > tol).sum().item()
        assert bad == 0, f'{name} {what}: {bad} of {err.numel()} outside tolerance, max err {err.max().item():.4g}'


def _model(seed, init):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    sd = synth.make_state_dict(seed, init)
    m = V2ce3d()
    m.load_state_dict(sd)
    return m.eval().to('cuda'), sd


@pytest.mark.parametrize('init,shape', [('lively', (1, 16, 2, 36, 44)), ('lively', (2, 16, 2, 20, 28)),
                                        ('reference', (1, 16, 2, 65, 87)), ('lively', (1, 16, 2, 260, 346))] +
                         # the other schedules: depth-merged at T=8 only, the seq_len % 8 != 0 schedule (direct head,
                         # gather, conv_halo T=2), three depth groups, the one-pixel bottleneck
                         [(init, shape) for shape in ((1, 8, 2, 40, 52), (2, 10, 2, 36, 44), (1, 24, 2, 36, 44),
                                                      (2, 16, 2, 8, 12)) for init in ('lively', 'reference')])
def test_forward_vs_fp32_oracle(init, shape):
    """Tolerance (stated, SURVEY.md F10): bf16 operands / fp32 accumulation / bf16 inter-layer activations against the
    fp32 reference, on two consecutive calls (spectral-norm state).  With the reference's own initialisation (what every
    other voxel test and the bench use) the calibrated bound holds with room: rel-L2 <= 1e-2, max-abs <= 3e-2 * max(ref)
    (measured on the B200: 4.2e-3 / 4.5e-3 at 65x87; 2.9e-3 / 3.4e-3 at 260x346 against cuDNN fp32,
    tests/test_gpu_torch_reference.py; cuDNN's own TF32 default deviates by 5.3e-4).  The 'lively' stress initialisation
    (He-scaled weights 8x the reference's, random BatchNorm statistics and biases: every layer carries signal and the
    bf16 rounding of 26 layers of activations accumulates, synth_inputs.make_state_dict) is
    measured at 0.92e-2 .. 1.31e-2 rel-L2 and 1.2e-2 .. 2.1e-2 max-abs depending on the plane size (gpurun_out/
    measurements_r2.jsonl, copied to profiles/voxel_tolerance_r2.jsonl): it is held to 1.6e-2 / 3e-2."""
    tol_rel, tol_max = (1e-2, 3e-2) if init == 'reference' else (1.6e-2, 3e-2)
    m, sd = _model(3, init)
    orc = UNetOracle(sd)
    g = torch.Generator(device='cpu').manual_seed(7)
    x = torch.randn(*shape, generator=g)
    for call in range(2):
        y = m(x.cuda()).cpu()
        ref = orc.forward(x)
        sig = m.last_sigmas()
        assert y.shape == ref.shape and (y >= 0).all()
        rel = float((y - ref).norm() / ref.norm())
        mx = float((y - ref).abs().max() / ref.abs().max())
        record_measurement('voxel_vs_fp32_oracle', init=init, shape=list(shape), call=call, rel_l2=rel, max_abs_over_max=mx)
        assert rel <= tol_rel and mx <= tol_max, (init, shape, call, rel, mx)
    assert m.call_count() == 2 and orc.calls == 2


def test_spectral_norm_schedule_matches_oracle():
    m, sd = _model(5, 'lively')
    orc = UNetOracle(sd)
    m.sn_advance(1)
    want = orc.sn_step()
    got = m.last_sigmas()
    assert np.allclose(got, np.array(want, dtype=np.float32), rtol=2e-5)
    m.sn_advance(3)
    for _ in range(3):
        want = orc.sn_step()
    assert np.allclose(m.last_sigmas(), np.array(want, dtype=np.float32), rtol=2e-5)


def test_forward_matches_reference_golden(golden, golden_meta):
    """Same inputs/weights the unmodified reference saw on CPU (tests/golden/make_golden.py)."""
    g = golden('unet')
    for name in ('refinit', 'lively'):
        meta = golden_meta['unet'][name]
        m, _ = _model(meta['seed'], meta['init'])
        x = torch.from_numpy(g[f'{name}_x']).cuda()
        for call in (0, 1):
            y = m(x).cpu().numpy()
            ref = g[f'{name}_y{call}']
            rel = np.linalg.norm(y - ref) / np.linalg.norm(ref)
            record_measurement('voxel_vs_reference_golden', name=name, call=call, rel_l2=float(rel),
                               max_abs_over_max=float(np.abs(y - ref).max() / np.abs(ref).max()))
            assert rel <= 1e-2, (name, call, rel)       # measured 2.9e-3 (reference init) / 7.9e-3 ('lively')


def test_rejects_cpu_input():
    from v2ce_toolbox_b200 import V2ceError
    m, _ = _model(0, 'reference')
    with pytest.raises(V2ceError):
        m(torch.zeros(1, 16, 2, 20, 28))


def test_forward_frames_equals_forward_of_preprocessed_units():
    """uint8 windows through the fused pre-processing == image_pre_processing (host, v2ce.py:45-64) + forward, bit for bit."""
    from v2ce_toolbox_b200.v2ce import image_pre_processing
    H, W = 36, 44
    frames = synth.make_video(35, H, W, seed=4)
    frames[0, 0, :4] = (0, 1, 254, 255)                      # the ends of the gray range
    # two 16-pair windows (tensor-pipe head) and one of 10 pairs (direct head, head_conv_kernel<true> against <false>)
    for wins in (np.stack([frames[0:17], frames[16:33]], axis=0), frames[None, 0:11]):
        units = torch.stack([image_pre_processing(w, H) for w in wins], dim=0)
        m1, _ = _model(2, 'lively')
        m2, _ = _model(2, 'lively')
        y_units = m1(units.cuda())
        y_frames = m2.forward_frames(torch.from_numpy(np.ascontiguousarray(wins)).cuda())
        assert torch.equal(y_units, y_frames), wins.shape


def test_full_size_batch_is_per_window_deterministic():
    """BASELINE configs[1] shape (batch 4, 346x260): every window of a batch equals the same window run alone, bit for
    bit (tiles never mix batch items; no atomics in the conv path), on two consecutive calls of the SN schedule."""
    for B, D, k in ((4, 16, 2), (3, 10, 1)):                 # (3, 10): the seq_len % 8 != 0 schedule
        mb, _ = _model(9, 'lively')
        m1, _ = _model(9, 'lively')
        g = torch.Generator(device='cpu').manual_seed(1)
        x = torch.randn(B, D, 2, 260, 346, generator=g).cuda()
        yb = mb(x)
        y1 = m1(x[k:k + 1].contiguous())
        assert torch.isfinite(yb).all() and (yb >= 0).all()
        assert torch.equal(yb[k:k + 1], y1), (B, D)
