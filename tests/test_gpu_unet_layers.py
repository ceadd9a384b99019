"""Per-layer parity of the V2ce3d forward on its real schedule, and the forward on a poisoned workspace.

Every conv layer, head and pred included, is run inside ``v2ce_model_forward`` with the model option ``stop_after``
(the forward returns right after the launch that writes that layer).  Every launch writes out of place, so the
workspace then holds the bf16 inputs the layer read and the output it wrote; the test recomputes the layer in fp64
from exactly those inputs and checks EVERY element against a bound derived from the operands:

    |got - ref| <= 2^-8 |ref| + 2^-16 S,    S = |scale| (|X| * |W|) + |shift terms| + |residual|

(* = the same conv on absolute values).  2^-8 is the bf16 rounding of the output; 2^-16 S leaves room for the fp32
accumulation order and the split-bf16 head and for nothing else.  With K = 27*768 products, dropping one K=16 step
moves a typical output by ~4/sqrt(K) = 3 % of |y|; the bound allows ~0.5 %.  test_bound_rejects_wrong_references
shows it: the same comparison against deliberately wrong references must fail.

Each row of ROWS exists to reach one branch of forward_impl (csrc/unet.cu); the launch count of a whole forward is
asserted so that a dispatch change cannot quietly move a row off that branch."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle.unet_oracle import UNetOracle, sn_conv_names
from conftest import record_measurement

pytestmark = pytest.mark.gpu

CH = (32, 64, 128, 256, 512)
# v2ce_model_workspace_layout order
BUFS = ('head_in', 'head', 'enc0', 'enc1', 'enc2', 'enc3', 'res0', 'res1', 'dec0', 'dec1', 'dec2', 'dec3',
        'tmp_t', 'tmp_r', 'up', 'up2')


def _layer_names():
    """kLayers of csrc/unet.cu (state-dict order): the index is the value of the option stop_after."""
    names = ['UNet.head.conv3d']
    blocks = [f'encoders.{i}' for i in range(4)] + [f'resblocks.{i}' for i in range(2)] + [f'decoders.{i}' for i in range(4)]
    for blk in blocks:
        names += [f'UNet.{blk}.conv1', f'UNet.{blk}.conv2', f'UNet.{blk}.downsample.0']
    return names + ['UNet.pred.conv3d']


LAYERS = _layer_names()
PRED = len(LAYERS) - 1
DEC3_CONV2 = LAYERS.index('UNet.decoders.3.conv2')

# B, D (seq_len), H, W, kernels of a whole forward (header of csrc/unet.cu: 30 at depth % 8 == 0; the other schedule
# runs the direct head (1), gather stride-2 convs and every shortcut unfused (4 x 3 + 2 x 3 + 4 x 3) = 35; at 8x12
# encoders.3 reads a one-row plane and falls back to two gather launches: 31)
ROWS = [
    pytest.param(1, 16, 260, 346, 30, id='cli_default_260x346'),         # T=16 head, stride-2 kdm, fused shortcuts
    pytest.param(1, 16, 1080, 346, 30, id='pano_h1080'),                 # tallest planes and their tile shapes
    pytest.param(3, 16, 65, 87, 30, id='odd_planes_b3'),                 # 65->33->17->9->5, upsample at non-2x ratios
    pytest.param(2, 16, 8, 12, 31, id='one_pixel_bottleneck'),           # encoders.3 on the gather kernel
    pytest.param(1, 8, 40, 52, 30, id='d8_kdm_t8'),                      # depth-merged kernel at T=8 only
    pytest.param(1, 24, 36, 44, 30, id='d24_three_groups'),              # three depth groups, no T=16
    pytest.param(2, 10, 36, 44, 35, id='d10_direct_head'),               # direct head, gather, conv_halo T=2, pred in conv_halo
    pytest.param(1, 9, 20, 28, 35, id='d9_halo_t1'),                     # the same schedule at T=1
]
U8_ROWS = ('cli_default_260x346', 'd10_direct_head')


def _levels(H, W):
    hs, ws = [H], [W]
    for _ in range(4):
        hs.append((hs[-1] - 1) // 2 + 1)
        ws.append((ws[-1] - 1) // 2 + 1)
    return hs, ws


def _schedule(li):
    """Where layer li reads and writes in the workspace (csrc/unet.cu forward_impl): sources [(buffer, level,
    channels)] in virtual-concat order, residual (buffer, level, channels) or None, output (buffer, level, channels,
    level it is stored nearest-upsampled to or None), stride, activation (1 relu).  Head and pred are special-cased."""
    _, blk, i, part = LAYERS[li].split('.', 3)
    i = int(i)
    conv2 = part == 'conv2'
    if blk == 'encoders':
        lo = i + 1
        src = [('tmp_t', lo, CH[lo])] if conv2 else [('head' if i == 0 else f'enc{i - 1}', i, CH[i])]
        out_buf = f'enc{i}' if conv2 else 'tmp_t' if part == 'conv1' else 'tmp_r'
        return src, ('tmp_r', lo, CH[lo]) if conv2 else None, (out_buf, lo, CH[lo], None), 1 if conv2 else 2
    if blk == 'resblocks':
        src = [('tmp_t', 4, 512)] if conv2 else [('enc3' if i == 0 else 'res0', 4, 512)]
        if conv2:
            out = ('res0', 4, 512, None) if i == 0 else ('up', 4, 512, 3)   # read only nearest-upsampled by decoders.0
        else:
            out = ('tmp_t' if part == 'conv1' else 'tmp_r', 4, 512, None)
        return src, ('tmp_r', 4, 512) if conv2 else None, out, 1
    lvl = 3 - i                                                              # decoders: output level
    if conv2:
        out = ('up2' if i % 2 == 0 else 'up', lvl, CH[lvl], lvl - 1) if lvl > 0 else None   # lvl 0: pred rides here
        return [('tmp_t', lvl, CH[lvl])], ('tmp_r', lvl, CH[lvl]), out, 1
    src = [('up' if i % 2 == 0 else 'up2', lvl, CH[lvl + 1]), ('head' if lvl == 0 else f'enc{lvl - 1}', lvl, CH[lvl])]
    return src, None, ('tmp_t' if part == 'conv1' else 'tmp_r', lvl, CH[lvl], None), 1


def _conv64(x, w, stride):
    """fp64 conv3d, padding k//2, stride (1, s, s); chunked over depth to bound cuDNN's working set."""
    p = w.shape[-1] // 2
    if p:
        x = F.pad(x, (p, p, p, p, p, p))
    D = x.shape[2] - 2 * p
    return torch.cat([F.conv3d(x[:, :, d0:d0 + 4 + 2 * p], w, None, (1, stride, stride)) for d0 in range(0, D, 4)], dim=2)


def _nearest_up(t, H, W):
    """NDHWC nearest upsample with the reference's (dst * in) // out indexing (unet_2layer.py:358-364)."""
    hi = (torch.arange(H, device=t.device) * t.shape[2]) // H
    wi = (torch.arange(W, device=t.device) * t.shape[3]) // W
    return t[:, :, hi][:, :, :, wi]


def _affine_ref(x, w, scale, shift, shift_mag, res, stride, act):
    """x (B,C,D,H,W) fp64 -> (y, S), both NDHWC fp64: y = act(scale * conv(x, w) + shift (+ res)), S its magnitude sum."""
    y = _conv64(x, w, stride) * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1)
    S = _conv64(x.abs(), w.abs(), stride) * scale.abs().view(1, -1, 1, 1, 1) + shift_mag.view(1, -1, 1, 1, 1)
    y, S = y.permute(0, 2, 3, 4, 1), S.permute(0, 2, 3, 4, 1)
    if res is not None:
        y = y + res
        S = S + res.abs()
    if act == 1:
        y = torch.relu(y)
    elif act == 2:
        y = F.leaky_relu(y, 0.01)
    return y, S


def _bound_check(got, ref, S):
    """(elements outside the bound, worst |got - ref| / bound); a NaN in `got` counts as outside."""
    err = (got.double() - ref).abs()
    bound = 2.0 ** -8 * ref.abs() + 2.0 ** -16 * S
    bad = int((~(err <= bound)).sum())
    worst = float(torch.nan_to_num(err / bound.clamp_min(1e-300), nan=float('inf')).max())
    return bad, worst


def _model(seed, init='lively'):
    from v2ce_toolbox_b200.scripts.v2ce_3d import V2ce3d
    sd = synth.make_state_dict(seed, init)
    m = V2ce3d()
    m.load_state_dict(sd)
    return m.eval().to('cuda'), sd


def _inputs(B, D, H, W, u8, seed=7):
    """(device input of the forward, fp32 image units the head sees) of one row."""
    if not u8:
        g = torch.Generator(device='cpu').manual_seed(seed)
        x = torch.randn(B, D, 2, H, W, generator=g)
        return x.cuda(), x.cuda()
    from v2ce_toolbox_b200.v2ce import image_pre_processing
    frames = synth.make_video(B * D + 1, H, W, seed=seed)
    wins = np.stack([frames[b * D:b * D + D + 1] for b in range(B)], axis=0)
    units = torch.stack([image_pre_processing(w, H) for w in wins], dim=0)
    return torch.from_numpy(wins).cuda(), units.cuda()


class Probe:
    """One model and one input of a row; runs the forward up to a layer and builds that layer's fp64 reference."""

    def __init__(self, B, D, H, W, u8=False):
        self.shape = (B, D, H, W)
        self.u8 = u8
        self.m, sd = _model(3)
        self.orc = UNetOracle(sd)
        self.x, self.units = _inputs(B, D, H, W, u8)
        self.hs, self.ws = _levels(H, W)
        lib = self.m._lib
        offs, n = (ctypes.c_int64 * len(BUFS))(), ctypes.c_int32()
        from v2ce_toolbox_b200._lib import check
        check(lib.v2ce_model_workspace_layout(self.m._handle, B, D, H, W, offs, len(BUFS), ctypes.byref(n)))
        assert n.value == len(BUFS)
        self.offsets = dict(zip(BUFS, offs[:]))

    def forward(self):
        return self.m.forward_frames(self.x) if self.u8 else self.m(self.x)

    def run(self, li):
        """Forward with stop_after = li on a workspace filled with 0xFF bytes (NaN in bf16): an output element the
        launch leaves unwritten fails the bound.  Returns (y, sigmas of this call)."""
        self.m.set_option('stop_after', li)
        try:
            if self.m._ws is None:
                self.forward()
            self.m._ws.fill_(0xFF)
            y = self.forward()
            return y, self.m.last_sigmas()
        finally:
            self.m.set_option('stop_after', -1)

    def view(self, buf, lvl, C, up_lvl=None):
        B, D = self.shape[:2]
        L = lvl if up_lvl is None else up_lvl
        n = B * D * self.hs[L] * self.ws[L] * C
        o = self.offsets[buf]
        return self.m._ws[o:o + 2 * n].view(torch.bfloat16).view(B, D, self.hs[L], self.ws[L], C)

    def _affine(self, name):
        """bf16-rounded weights as packed (weight_bar for SN layers), BN folded as in v2ce_model_finalize:
        (w, scale without 1/sigma, shift, magnitude sum of the shift's terms), fp64 on the device."""
        o = self.orc
        w = o._conv_weight(name, {name: 1.0}).to(torch.bfloat16).double().cuda()
        if name.endswith('downsample.0'):
            bn, bias = name[:-2] + '.1', o.sd[name + '.bias'].double()
        else:
            bn, bias = name.replace('.conv', '.bn'), None
        s, _ = o._bn_fold(bn)
        s = s.double()
        b, mu = o.sd[bn + '.bias'].double(), o.sd[bn + '.running_mean'].double()
        shift, mag = b - mu * s, b.abs() + (mu * s).abs()
        if bias is not None:
            shift, mag = shift + bias * s, mag + (bias * s).abs()
        return w, s.cuda(), shift.cuda(), mag.cuda()

    def check(self, li, mutate=None):
        """Run up to layer li and compare; `mutate` ('drop_k', 'shift_up', 'swap_concat') falsifies the reference
        only.  Returns (bad elements, worst ratio, elements checked)."""
        y, sig = self.run(li)
        sigma = dict(zip(sn_conv_names(), sig))
        if li == 0:
            wt = self.orc.sd['UNet.head.conv3d.weight'].double().cuda()
            if mutate == 'drop_k':
                wt[:, :, 1, 1, 1] = 0
            bias = self.orc.sd['UNet.head.conv3d.bias'].double().cuda()
            x = self.units.double().permute(0, 2, 1, 3, 4)
            ref, S = _affine_ref(x, wt, torch.ones_like(bias), bias, bias.abs(), None, 1, 2)
            return (*_bound_check(self.view('head', 0, 32), ref, S), ref.numel())
        if li in (DEC3_CONV2, PRED):
            name = LAYERS[DEC3_CONV2]
        else:
            name = LAYERS[li]
        srcs, res, out, stride = _schedule(LAYERS.index(name))
        up_store = out is not None and out[3] is not None
        w, s, shift, mag = self._affine(name)
        if name in sigma:
            s = s / float(sigma[name])
        xs = [self.view(b, lv, c).double() for b, lv, c in srcs]
        if mutate == 'swap_concat':
            xs = xs[::-1]
        if mutate == 'shift_up' and not up_store:                 # the nearest-upsampled decoder input
            xs[0] = torch.roll(xs[0], 1, dims=2)
        if mutate == 'drop_k' and li != PRED:
            w[:, :16, w.shape[2] // 2, w.shape[3] // 2, w.shape[4] // 2] = 0
        x = torch.cat(xs, dim=-1).permute(0, 4, 1, 2, 3)
        r = self.view(*res).double() if res is not None else None
        ref, S = _affine_ref(x, w, s, shift, mag, r, stride, 1 if name.endswith(('conv1', 'conv2')) else 0)
        if li in (DEC3_CONV2, PRED):
            # pred rides in decoders.3.conv2, which keeps its result in fp32: relu(Wp . y32 + bp), magnitudes carried
            wp = self.orc.sd['UNet.pred.conv3d.weight'].double().cuda().view(20, 32)
            bp = self.orc.sd['UNet.pred.conv3d.bias'].double().cuda()
            if mutate == 'drop_k':
                wp[:, :16] = 0
            ref = torch.relu(ref @ wp.t() + bp).permute(0, 1, 4, 2, 3)
            S = (S @ wp.abs().t() + bp.abs()).permute(0, 1, 4, 2, 3)
            return (*_bound_check(y, ref, S), ref.numel())
        got = self.view(*out)
        if up_store:
            L = out[3]
            ref, S = _nearest_up(ref, self.hs[L], self.ws[L]), _nearest_up(S, self.hs[L], self.ws[L])
            if mutate == 'shift_up':
                ref = torch.roll(ref, 1, dims=2)
        return (*_bound_check(got, ref, S), ref.numel())


@pytest.mark.parametrize('B,D,H,W,launches', ROWS)
def test_every_layer_within_operand_bound(B, D, H, W, launches, request):
    row = request.node.callspec.id
    with torch.no_grad():
        p = Probe(B, D, H, W)
        p.forward()
        assert p.m.last_launches() == launches
        failures = []
        for li in range(len(LAYERS)):
            bad, worst, n = p.check(li)
            record_measurement('unet_layer_bound', row=row, layer=LAYERS[li], worst_ratio=worst, elements=n)
            if bad:
                failures.append(f'{LAYERS[li]}: {bad} of {n} outside the bound')
        assert not failures, failures
        if row in U8_ROWS:
            # the uint8 entry differs from the fp32 one only in the head's input (the fused pre-processing)
            p = Probe(B, D, H, W, u8=True)
            p.forward()
            assert p.m.last_launches() == launches
            bad, worst, n = p.check(0)
            record_measurement('unet_layer_bound', row=row + '_u8', layer=LAYERS[0], worst_ratio=worst, elements=n)
            assert bad == 0, f'uint8 head: {bad} of {n} outside the bound'


@pytest.mark.parametrize('B,D,H,W,launches', ROWS)
def test_forward_on_poisoned_workspace(B, D, H, W, launches, request):
    """Twin models (same seed, first call) through the C ABI: workspace 0xFF bytes (NaN in bf16 and fp32) and y
    NaN-filled, against both zero-filled.  The outputs must be finite and bitwise equal: no element is left unwritten
    and nothing is multiplied out of never-written memory (the tail of the overlapping-row views of the 32-channel
    tensors, K steps beyond the real channels).  The caching allocator can hand out such bit patterns."""
    from v2ce_toolbox_b200._lib import check, ptr, stream_ptr
    for u8 in ((False, True) if request.node.callspec.id in U8_ROWS else (False,)):
        x, _ = _inputs(B, D, H, W, u8)
        ys = []
        for fill in (0xFF, 0):
            m, _ = _model(5)
            n = ctypes.c_size_t()
            check(m._lib.v2ce_model_workspace_bytes(m._handle, B, D, H, W, ctypes.byref(n)))
            ws = torch.full((n.value,), fill, dtype=torch.uint8, device='cuda')
            y = torch.full((B, D, 20, H, W), float('nan') if fill else 0.0, device='cuda')
            fn = m._lib.v2ce_model_forward_frames if u8 else m._lib.v2ce_model_forward
            check(fn(m._handle, ptr(x), ptr(y), B, D, H, W, ptr(ws), n.value, stream_ptr()))
            torch.cuda.synchronize()
            assert m.last_launches() == launches
            ys.append(y)
        assert torch.isfinite(ys[0]).all(), f'u8={u8}: {int((~torch.isfinite(ys[0])).sum())} non-finite outputs'
        assert torch.equal(ys[0], ys[1]), f'u8={u8}: outputs depend on the workspace contents'


# one layer of each kernel family on the odd-plane row, with the mutations that apply to it
MUTATIONS = [
    ('UNet.head.conv3d', 'drop_k'),                  # head: split-bf16 pixels on the depth-merged kernel
    ('UNet.encoders.1.conv1', 'drop_k'),             # depth-merged, stride 2, fused shortcut
    ('UNet.decoders.3.conv1', 'drop_k'),             # depth-merged, two sources, 32-channel dense skip
    ('UNet.decoders.3.conv1', 'shift_up'),
    ('UNet.decoders.3.conv1', 'swap_concat'),
    ('UNet.decoders.2.conv2', 'shift_up'),           # depth-merged, upsample-on-store
    ('UNet.decoders.0.conv1', 'drop_k'),             # halo, K = 27 * 768
    ('UNet.decoders.0.conv1', 'shift_up'),
    ('UNet.decoders.0.conv1', 'swap_concat'),
    ('UNet.resblocks.1.conv2', 'shift_up'),          # halo, upsample-on-store
    ('UNet.decoders.1.downsample.0', 'drop_k'),      # gather (side stream)
    ('UNet.decoders.1.downsample.0', 'shift_up'),
    ('UNet.decoders.1.downsample.0', 'swap_concat'),
    ('UNet.pred.conv3d', 'drop_k'),                  # pred fused into decoders.3.conv2
]


def test_bound_rejects_wrong_references():
    """The per-layer bound can fail: the comparison against a deliberately wrong reference (one K=16 channel step of
    one tap dropped, the upsampled tensor shifted by one row, the two concat sources swapped) reports mismatches.
    Only the reference is altered, never a kernel."""
    with torch.no_grad():
        p = Probe(3, 16, 65, 87)
        accepted = []
        for name, mutate in MUTATIONS:
            bad, _, n = p.check(LAYERS.index(name), mutate)
            record_measurement('unet_layer_bound_mutation', layer=name, mutation=mutate, rejected=bad, elements=n)
            if bad == 0:
                accepted.append((name, mutate))
        assert not accepted, f'wrong references accepted: {accepted}'
