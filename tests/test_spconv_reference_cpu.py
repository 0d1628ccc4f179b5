"""The float64 reference of tests/test_gpu_spconv.py is the operation it claims to be: it equals the oracle's spconv
'native' form (oracle.sparse_conv_mm) on random neighbour tables and a dense conv3d on a fully occupied grid."""
import numpy as np
import torch

from oracle import oracle
from test_gpu_spconv import BF16X2, F16, F16X2, F32, exact_mask, reference, split_parts, table
from util import nbr_to_pairs


def test_reference_equals_sparse_conv_mm():
    g = torch.Generator().manual_seed(0)
    n_in, cap, n_out, cin, cout, kvol = 300, 256, 201, 8, 16, 27
    x = torch.randn(n_in, cin, generator=g)
    w = torch.randn(kvol, cin, cout, generator=g)
    bias = torch.randn(cout, generator=g)
    nbr = table('random', kvol, cap, n_in, g, 0.4)
    ref, s = reference(x, w, nbr, n_out, F32, bias)
    want = oracle.sparse_conv_mm(x.numpy(), w.numpy(), nbr_to_pairs(nbr.numpy(), n_out), n_out) + bias.numpy()
    np.testing.assert_allclose(ref.numpy(), want, rtol=1e-5, atol=1e-5)
    assert (s >= ref.abs() - 1e-9).all()
    res = torch.randn(cap, cout, generator=g, dtype=torch.float64)
    ref2, _ = reference(x, w, nbr, n_out, F32, bias, res, relu=True)
    np.testing.assert_allclose(ref2.numpy(), np.maximum(want + res[:n_out].numpy(), 0), rtol=1e-5, atol=1e-5)


def test_reference_equals_conv3d():
    g = torch.Generator().manual_seed(1)
    D, H, W, cin, cout = 4, 5, 6, 3, 5
    x = torch.randn(1, cin, D, H, W, generator=g, dtype=torch.float64)
    wt = torch.randn(cout, cin, 3, 3, 3, generator=g, dtype=torch.float64)
    cells = torch.arange(D * H * W)
    z, y, xx = cells // (H * W), (cells // W) % H, cells % W
    cap = 128
    nbr = torch.full((27, cap), -1, dtype=torch.int32)
    for k in range(27):
        iz, iy, ix = z - 1 + k // 9, y - 1 + (k // 3) % 3, xx - 1 + k % 3
        ok = (iz >= 0) & (iz < D) & (iy >= 0) & (iy < H) & (ix >= 0) & (ix < W)
        nbr[k, cells[ok]] = ((iz * H + iy) * W + ix)[ok].to(torch.int32)
    rows = x[0].permute(1, 2, 3, 0).reshape(-1, cin)
    w_kio = wt.permute(2, 3, 4, 1, 0).reshape(27, cin, cout)
    ref, _ = reference(rows.float(), w_kio.float(), nbr, D * H * W, F32)
    want = torch.nn.functional.conv3d(rows.float().double().reshape(1, D, H, W, cin).permute(0, 4, 1, 2, 3),
                                      w_kio.float().double().reshape(3, 3, 3, cin, cout).permute(4, 3, 0, 1, 2), padding=1)
    np.testing.assert_allclose(ref.numpy(), want[0].permute(1, 2, 3, 0).reshape(-1, cout).numpy(), rtol=1e-12, atol=1e-12)


def test_reference_split_products_and_masks():
    """Split operands: the reference sums exactly xh.Wh + xl.Wh + xh.Wl; exact tile masks follow the header's definition."""
    g = torch.Generator().manual_seed(2)
    x, w = torch.randn(50, 16, generator=g), torch.randn(3, 16, 8, generator=g)
    nbr = table('random', 3, 128, 50, g, 0.6)
    for enc in (F16X2, BF16X2):
        xh, xl = (t.double() for t in split_parts(x, enc))
        wh, wl = (t.double() for t in split_parts(w, enc))
        assert ((xh + xl - x.double()).abs() <= x.double().abs() * 2.0 ** -16 + 2.0 ** -25).all()   # (f16: subnormal lo)
        ref, _ = reference(x, w, nbr, 128, enc)
        want = torch.zeros(128, 8, dtype=torch.float64)
        for k in range(3):
            for o in range(128):
                i = int(nbr[k, o])
                if i >= 0:
                    want[o] += xh[i] @ wh[k] + xl[i] @ wh[k] + xh[i] @ wl[k]
        np.testing.assert_allclose(ref.numpy(), want.numpy(), rtol=1e-12, atol=1e-12)
    hi, lo = split_parts(torch.tensor([1.0e5, 3.0e-8]), F16)
    assert hi.tolist() == [65504.0, float(torch.tensor(3.0e-8).half())] and lo.tolist() == [0.0, 0.0]
    nbr = torch.full((5, 384), -1, dtype=torch.int32)
    nbr[1, 5] = 0
    nbr[3, 130] = 7
    nbr[4, 300] = 2            # past n_out: not in the mask
    assert exact_mask(nbr, 290, 384).tolist() == [2, 8, 0]
