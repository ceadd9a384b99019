"""Bring-up helper: run ONE conv case of tests/test_gpu_unet.py in its own process and print error structure."""
import sys
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests'))
import numpy as np
import torch
import test_gpu_unet as T


def main(name, impl=0):
    case = [c for c in T.CASES + T.HALO_CASES + T.KDM_CASES if c[0] == name][0]
    _, B, D, hin, win, C0, up, C1, cout, k, stride, use_res, act = case
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
    try:
        out = T.conv_hook(src0, src1, hin, win, w, scale, shift, res, act, k, stride, impl=impl)
    except Exception as e:
        print(f'CASE {name}: EXCEPTION {e}')
        return 2
    ref = T.torch_ref(src0, src1, hin, win, w, scale, shift, res, act, k, stride)
    o = out.float().reshape(-1, cout)
    r = ref.reshape(-1, cout)
    nan = torch.isnan(o).sum().item()
    err = (o - r).abs()
    err[torch.isnan(err)] = 1e9
    tol = 2.0 ** -8 * r.abs() + 2e-3
    bad = err > tol
    print(f'CASE {name} impl={impl}: M={o.shape[0]} N={cout} K={cin * k ** 3} nan={nan} bad={bad.sum().item()}/{bad.numel()} '
          f'maxerr={err[~torch.isnan(o)].max().item() if nan < o.numel() else -1:.4g} refmax={r.abs().max().item():.3g}')
    if bad.any():
        rows = bad.any(dim=1).nonzero().flatten()
        cols = bad.any(dim=0).nonzero().flatten()
        print('  bad rows (first 24):', rows[:24].tolist(), ' count', rows.numel())
        print('  bad cols (first 24):', cols[:24].tolist(), ' count', cols.numel())
        idx = bad.nonzero()[:6]
        for m, n in idx.tolist():
            print(f'   m={m} n={n} got={o[m, n].item():.5f} ref={r[m, n].item():.5f}')
        return 1
    return 0


if __name__ == '__main__':
    sys.exit(main(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 0))
