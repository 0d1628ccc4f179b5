"""Layer-level tests of the sparse-convolution kernels against a float64 reference of the same operation.

srf_spconv_tc (tcgen05 gather-GEMM, and the warp-MMA 16 -> 16 kernel it dispatches to), srf_spconv_f32 (SIMT), the
dense-rulebook path of the BEV convolutions and srf_convert_rows, at the shapes, encodings and edges where a kernel goes
wrong: every channel pair of the dispatch table in every operand encoding, every output encoding, kvol 27 / 9 / 3 / 1,
tile masks (none, exact, over-set, a live tile without neighbours), partial offset groups, ragged device-side row counts
with a sentinel past the count, persistent grids of three or more tiles per CTA, dense scatter, residual and ReLU.

Bound (elementwise, never a global max-relative error, which hides errors in small rows):

    |got - ref| <= EPS_ACC * S + eps_out(out) * |ref| + floor(out)

ref is float64 over the values the kernel multiplies (rounded plain operands, or the three products xh.Wh + xl.Wh + xh.Wl
of the split operands, hi = round16(v), lo = round16(v - hi), built in torch), so what is left is fp32 accumulation and
output rounding.  S = sum |x||W| + |bias| + |residual| per output element.  eps_out is the output format's half-ulp and
floor its half subnormal spacing (f16 forms).

EPS_ACC: calibrated on an NVIDIA B200 (1000 W power limit) with the whole file.  The largest observed
(|got - ref| - eps_out |ref| - floor) / S, per input encoding, was for tcgen05: f16 6.9e-7, bf16 5.9e-7, bf16x2 1.7e-6,
f16x2 2.1e-6 (f16x2 -> f16x2); for the SIMT kernel: f32 3.9e-7, bf16 3.6e-7.  EPS_TC / EPS_SIMT are 4x the largest
(RATIO_* below).  The file runs in about 20 s on that B200.
"""
import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F32, BF16, F16, BF16X2, F16X2 = 0, 1, 2, 3, 4      # include/srfdet_b200.h element encodings
ENC = {'f32': F32, 'bf16': BF16, 'f16': F16, 'bf16x2': BF16X2, 'f16x2': F16X2}
SPLIT = (BF16X2, F16X2)
ERR_ARG, ERR_UNSUPPORTED = -1, -3

RATIO_TC = 2.2e-6      # largest observed ratio, all tcgen05 cases (f16x2 -> f16x2)
RATIO_SIMT = 4.0e-7    # largest observed ratio, all SIMT cases (f32 -> f32)
EPS_TC = 4 * RATIO_TC
EPS_SIMT = 4 * RATIO_SIMT
EPS_OUT = {F32: 0.0, F16: 2.0 ** -11, BF16: 2.0 ** -8, F16X2: 2.0 ** -22, BF16X2: 2.0 ** -17}
FLOOR = {F32: 0.0, F16: 2.0 ** -25, BF16: 0.0, F16X2: 2.0 ** -25, BF16X2: 0.0}

# channel pairs of dispatch_sparse (igemm_umma.cu) plus column-tiled outputs (n_tiles 2 and 3)
TC_PAIRS = [(16, 16), (16, 32), (32, 32), (32, 64), (64, 64), (64, 128), (128, 128), (128, 64), (64, 32), (32, 16),
            (256, 128), (256, 64), (128, 256), (128, 384), (256, 256), (256, 384)]
ENCS = ['f16', 'bf16', 'f16x2', 'bf16x2']

_ratios = {}


# ------------------------------------------------------------------------------------------------ encodings / reference
def is_f16(enc):
    return enc in (F16, F16X2)


def round16(v, f16):
    """fp32 -> nearest 16-bit value as fp32 (f16 saturates at +-65504 like the kernels' stores)."""
    v = v.float()
    if f16:
        return v.clamp(-65504.0, 65504.0).half().float()
    return v.bfloat16().float()


def split_parts(v, enc):
    """The values a kernel sees for encoding enc: (hi, lo) fp32 tensors (lo = 0 for plain forms, hi = v for f32)."""
    v = v.float()
    if enc == F32:
        return v, torch.zeros_like(v)
    hi = round16(v, is_f16(enc))
    lo = round16(v - hi, is_f16(enc)) if enc in SPLIT else torch.zeros_like(v)
    return hi, lo


def encode(v, enc):
    """(rows, c) fp32 -> the buffer of encoding enc, built in torch (split rows [hi | lo])."""
    if enc == F32:
        return v.float().contiguous()
    dt = torch.float16 if is_f16(enc) else torch.bfloat16
    hi, lo = split_parts(v, enc)
    if enc in SPLIT:
        return torch.cat([hi, lo], 1).to(dt).contiguous()
    return hi.to(dt).contiguous()


def decode(t, c):
    if t.dtype != torch.float32 and t.shape[-1] == 2 * c:
        return t[..., :c].double() + t[..., c:].double()
    return t.double()


def reference(x, w, nbr, n_out, in_enc, bias=None, residual=None, relu=False, w_enc=None):
    """float64 out[o] = act(sum_k W_k^T x[nbr[k][o]] + bias (+ residual[o])) over rows o < n_out, on x's device.

    x (n_in, cin) and w (kvol, cin, cout) fp32 values; in_enc / w_enc say what the kernel multiplies: the rounded plain
    operands, or for the split forms the three products xh.Wh + xl.Wh + xh.Wl; SRF_F32 multiplies the fp32 values.
    residual: decoded values (float64) or None.  Returns (ref, S) with S = sum |x||W| + |bias| + |residual|."""
    w_enc = in_enc if w_enc is None else w_enc
    xh, xl = (t.double() for t in split_parts(x, in_enc))
    wh, wl = (t.double() for t in split_parts(w, w_enc))
    kvol, cin, cout = w.shape
    nb = nbr[:, :n_out].long()
    ref = torch.zeros((n_out, cout), dtype=torch.float64, device=x.device)
    s = torch.zeros_like(ref)
    for k in range(kvol):
        idx = nb[k]
        ok = (idx >= 0).double()[:, None]
        ih = xh[idx.clamp(min=0)] * ok
        ref += ih @ wh[k]
        s += ih.abs() @ wh[k].abs()
        if in_enc in SPLIT:
            il = xl[idx.clamp(min=0)] * ok
            ref += il @ wh[k] + ih @ wl[k]
    if bias is not None:
        ref += bias.double()
        s += bias.double().abs()
    if residual is not None:
        ref += residual[:n_out]
        s += residual[:n_out].abs()
    if relu:
        ref = torch.relu(ref)
    return ref, s


def check_bound(got, ref, s, out_enc, eps_acc, tag, key=None):
    """Elementwise bound; records the case's largest ratio under key (kernel, in encoding, out encoding)."""
    got = got.double()
    err = (got - ref).abs()
    slack = EPS_OUT[out_enc] * ref.abs() + FLOOR[out_enc]
    ratio = ((err - slack) / s.clamp(min=1e-30)).max().item() if err.numel() else 0.0
    if key is not None:
        _ratios[key] = max(_ratios.get(key, -1.0), ratio)
    bad = err > eps_acc * s + slack
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError(f'{tag}: {int(bad.sum())} elements out of bound; first {i}: got {got[tuple(i)].item():.9g} '
                             f'ref {ref[tuple(i)].item():.9g} S {s[tuple(i)].item():.3g} ratio {ratio:.3g}')
    assert torch.isfinite(got).all(), tag


def _lib():
    from srfdet_b200 import _lib as L
    return L, L.load()


def _ptr(t):
    return None if t is None else t.data_ptr()


def exact_mask(nbr, n_out, cap):
    """tile_mask[t] bit k set iff some row < n_out of tile t has a neighbour at k (include/srfdet_b200.h)."""
    kvol = nbr.shape[0]
    has = (nbr[:, :cap] >= 0).clone()
    has[:, n_out:] = False
    per_tile = has.view(kvol, cap // 128, 128).any(2).long()                         # (kvol, tiles)
    bits = (per_tile << torch.arange(kvol, device=nbr.device)[:, None]).sum(0)
    return bits.to(torch.int64).to(torch.int32).contiguous()                         # bit 31 unused (kvol <= 27)


# ------------------------------------------------------------------------------------------------ neighbour tables
def table(pattern, kvol, cap, n_in, g, density=0.5):
    if pattern == 'random':
        nbr = torch.randint(0, n_in, (kvol, cap), generator=g, dtype=torch.int32)
        nbr[torch.rand(kvol, cap, generator=g) >= density] = -1
    elif pattern == 'banded':       # SubM-like: row o reads inputs near o * n_in / cap, centre always present
        base = (torch.arange(cap, dtype=torch.int64) * n_in // cap)[None, :]
        nbr = (base + torch.randint(-60, 60, (kvol, cap), generator=g)).clamp_(0, n_in - 1).to(torch.int32)
        nbr[torch.rand(kvol, cap, generator=g) >= density] = -1
        nbr[kvol // 2] = base[0].to(torch.int32)
    elif pattern == 'hub':          # one input row feeds many outputs through many offsets
        nbr = torch.randint(0, n_in, (kvol, cap), generator=g, dtype=torch.int32)
        nbr[torch.rand(kvol, cap, generator=g) < 0.6] = n_in // 3
        nbr[torch.rand(kvol, cap, generator=g) < 0.2] = -1
    elif pattern == 'last':         # the last input row, everywhere it can be
        nbr = torch.randint(0, n_in, (kvol, cap), generator=g, dtype=torch.int32)
        nbr[torch.rand(kvol, cap, generator=g) < 0.5] = n_in - 1
        nbr[torch.rand(kvol, cap, generator=g) < 0.2] = -1
    else:
        raise ValueError(pattern)
    return nbr


# ------------------------------------------------------------------------------------------------ srf_spconv_tc runner
def run_tc(cin, cout, enc, out_enc=None, kvol=27, cap=1024, n_out='ragged', n_in=3000, pattern='random', density=0.5,
           mask='none', residual=False, relu=True, seed=0, nbr=None, bias=None, check=True, tag=''):
    """One srf_spconv_tc call on a seeded problem; checks the bound and the sentinel past the count.
    n_out: an int (device count), None (no count: all cap rows) or 'ragged' (cap - 37).
    mask: 'none' | 'exact' | 'ones' | a (cap // 128) int32 tensor."""
    L, lib = _lib()
    out_enc = enc if out_enc is None else out_enc
    g = torch.Generator().manual_seed(seed)
    live = cap - 37 if n_out == 'ragged' else (cap if n_out is None else n_out)
    x = torch.randn(n_in, cin, generator=g).cuda()
    w = (torch.randn(kvol, cin, cout, generator=g) / (kvol * cin / 3) ** 0.5).cuda()
    bias = (torch.randn(cout, generator=g) * 0.5).cuda() if bias is None else bias.cuda()
    if nbr is None:
        nbr = table(pattern, kvol, cap, n_in, g, density)
    nbr = nbr.cuda().contiguous()
    res_t = encode((torch.randn(cap, cout, generator=g) * 0.5).cuda(), out_enc) if residual else None
    xe = _convert(x, enc)
    wp = torch.empty(L.enc_width(enc, kvol * cin * cout), dtype=L.enc_torch_dtype(enc), device='cuda')
    st = L.stream_ptr()
    L.check(lib.srf_pack_weight_tc(_ptr(w), kvol, cin, cout, enc, _ptr(wp), st), 'pack')
    if isinstance(mask, torch.Tensor):
        tm = mask.cuda().contiguous()
    elif mask == 'exact':
        tm = exact_mask(nbr, live, cap)
    elif mask == 'ones':
        tm = torch.full((cap // 128,), -1, dtype=torch.int32, device='cuda')
    else:
        tm = None
    cnt = None if n_out is None else torch.tensor([live], dtype=torch.int32, device='cuda')
    width = L.enc_width(out_enc, cout)
    out = torch.empty((cap, width), dtype=L.enc_torch_dtype(out_enc), device='cuda')
    out.view(torch.int16 if out.dtype != torch.float32 else torch.int32).fill_(0x3F1B)      # sentinel bit pattern
    sentinel = out.clone()
    a = L.ConvArgs()
    a.in_, a.in_dtype, a.in_rows = _ptr(xe), enc, n_in
    a.cin, a.cout, a.kvol = cin, cout, kvol
    a.nbr, a.tile_mask, a.cap_out, a.d_n_out = _ptr(nbr), _ptr(tm), cap, _ptr(cnt)
    a.w, a.bias, a.residual, a.relu = _ptr(wp), _ptr(bias), _ptr(res_t), int(relu)
    a.out, a.out_dtype = _ptr(out), out_enc
    L.check(lib.srf_spconv_tc(ctypes.byref(a), st), f'srf_spconv_tc {tag}')
    torch.cuda.synchronize()
    res = decode(res_t, cout) if residual else None
    ref, s = reference(x, w, nbr, live, enc, bias, res, relu)
    got = decode(out[:live], cout)
    if check:
        what = f'tc {cin}->{cout} {enc}->{out_enc} {tag}'
        check_bound(got, ref, s, out_enc, EPS_TC, what, ('tc', enc, out_enc))
        assert torch.equal(out[live:], sentinel[live:]), 'rows past the count were written'
        if enc in SPLIT:
            # end to end against the unrounded fp32 operands: the split products are exact to 2^-16 (bf16) / 2^-21 (f16)
            ref32, s32 = reference(x, w, nbr, live, F32, bias, res, relu)
            prod = 2.0 ** -21 if is_f16(enc) else 2.0 ** -16
            check_bound(got, ref32, s32, out_enc, 2 * prod + EPS_TC, what + ' vs fp32 operands')
    return dict(got=got, ref=ref, s=s, live=live, out=out)


def _convert(x, enc):
    """The library's srf_convert_rows (what the model feeds its convolutions); its encoding is pinned bit for bit below."""
    L, lib = _lib()
    out = torch.empty((x.shape[0], L.enc_width(enc, x.shape[1])), dtype=L.enc_torch_dtype(enc), device='cuda')
    L.check(lib.srf_convert_rows(_ptr(x.contiguous()), x.shape[0], x.shape[1], x.shape[1], enc, _ptr(out), L.stream_ptr()),
            'convert')
    return out


# ------------------------------------------------------------------------------------------------ srf_spconv_tc matrix
@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('cin,cout', TC_PAIRS)
def test_tc_channel_pairs(cin, cout, enc):
    """Every template configuration (channel pair x plain / split), same-encoding output, residual + ReLU."""
    run_tc(cin, cout, ENC[enc], residual=True, relu=True, seed=cin * 7 + cout)


@pytest.mark.parametrize('enc', ['f16', 'bf16x2'])
@pytest.mark.parametrize('cin,cout', TC_PAIRS)
def test_tc_persistent_loop(cin, cout, enc):
    """At least 3 * 2 * sm_count * 128 rows: every CTA of the persistent grid runs three or more tiles, so the TMEM
    double buffer, the ring-phase wraparound and the one-tile-ahead index prefetch run many times."""
    L, lib = _lib()
    cap = 3 * 2 * lib.srf_sm_count() * 128 + 5 * 128
    out = F32 if (cin, cout) == (16, 16) and ENC[enc] not in SPLIT else ENC[enc]      # (same-encoding 16 -> 16: warp kernel)
    run_tc(cin, cout, ENC[enc], out, cap=cap, n_in=40000, density=0.3, residual=(cout <= 128), relu=False, mask='exact',
           seed=cin + cout)


@pytest.mark.parametrize('cin,cout', [(32, 64), (256, 384), (16, 16)])
@pytest.mark.parametrize('enc,out', [('f16', 'f32'), ('bf16', 'f32'), ('f16x2', 'f32'), ('bf16x2', 'f32'),
                                     ('f16x2', 'f16'), ('bf16x2', 'bf16'), ('f16', 'f16x2'), ('bf16', 'bf16x2')])
def test_tc_output_encodings(cin, cout, enc, out):
    """Outputs in F32, split in -> plain out, plain in -> split out, each with a residual in the output encoding."""
    for relu in (False, True):
        run_tc(cin, cout, ENC[enc], ENC[out], residual=True, relu=relu, seed=3 + relu)


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('kvol', [27, 9, 3, 1])
def test_tc_kernel_sizes(kvol, enc):
    for cin, cout in [(16, 32), (64, 64), (256, 128), (128, 256)]:
        run_tc(cin, cout, ENC[enc], kvol=kvol, mask='exact', residual=(kvol == 3), relu=(kvol != 9), seed=kvol,
               tag=f'kvol {kvol}')
    run_tc(16, 16, ENC[enc], F32, kvol=kvol, seed=kvol, tag=f'16->16 f32 out, kvol {kvol}')


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('mask', ['none', 'exact', 'ones'])
def test_tc_tile_masks(mask, enc):
    for cin, cout in [(16, 32), (64, 128), (256, 128)]:
        run_tc(cin, cout, ENC[enc], kvol=27, mask=mask, pattern='banded', density=0.3, residual=True, seed=5, tag=mask)


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('cin,cout', [(16, 32), (32, 32), (64, 128), (256, 384)])
def test_tc_empty_tiles(cin, cout, enc):
    """Live tiles with no neighbour at all and tile_mask 0: their rows are act(bias + residual).  The table is large enough
    that every CTA runs several tiles, so an empty tile follows tiles that left an accumulator in its TMEM buffer."""
    L, lib = _lib()
    cap = 3 * 2 * lib.srf_sm_count() * 128 + 4 * 128
    g = torch.Generator().manual_seed(17)
    nbr = table('random', 27, cap, 20000, g, 0.4)
    tiles = cap // 128
    empty = torch.zeros(tiles, dtype=torch.bool)
    empty[3::5] = True
    empty[-2] = True                                            # the last full tile too
    nbr.view(27, tiles, 128)[:, empty] = -1
    live = cap - 100
    tm = exact_mask(nbr.cuda(), live, cap)
    assert (tm.cpu()[empty] == 0).all() and (tm.cpu()[~empty] != 0).all()
    for relu in (False, True):
        r = run_tc(cin, cout, ENC[enc], cap=cap, n_out=live, n_in=20000, nbr=nbr, mask=tm, residual=True, relu=relu,
                   seed=1 + int(relu), tag='empty tiles')
        rows = empty.repeat_interleave(128)[:live].cuda()
        assert (r['got'][rows] != 0).any()                      # act(bias + residual) is not trivially zero


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('cout', [16, 32])
def test_tc_partial_offset_groups(cout, enc):
    """cin 16 carries G = 4 (plain) / 2 (split) kernel offsets per ring slot: tiles with 1, 2, 3, 5, 6 and 7 active offsets
    leave the last group partly filled.  (16 -> 16 with an f32 output runs the tcgen05 kernel.)"""
    cap, n_in = 6 * 128 * 4, 5000
    g = torch.Generator().manual_seed(23 + cout)
    nbr = table('random', 27, cap, n_in, g, 0.7)
    counts = [1, 2, 3, 5, 6, 7]
    for t in range(cap // 128):
        keep = torch.zeros(27, dtype=torch.bool)
        keep[torch.randperm(27, generator=g)[:counts[t % 6]]] = True
        nbr[~keep, t * 128:(t + 1) * 128] = -1
    out = F32 if cout == 16 else ENC[enc]
    run_tc(16, cout, ENC[enc], out, cap=cap, n_in=n_in, nbr=nbr, mask='exact', residual=True, seed=cout, tag='groups')


@pytest.mark.parametrize('enc', ['f16', 'bf16x2'])
@pytest.mark.parametrize('n_out', [0, 1, 127, 128, 129, 1023, 1024, None])
def test_tc_row_counts(n_out, enc):
    for cin, cout in [(64, 128), (256, 256)]:
        run_tc(cin, cout, ENC[enc], cap=1024, n_out=n_out, mask='exact', residual=True, seed=7, tag=f'n_out {n_out}')


@pytest.mark.parametrize('enc', ['bf16', 'f16x2'])
@pytest.mark.parametrize('pattern,density', [('random', 0.5), ('banded', 3.7 / 27), ('banded', 15 / 27), ('hub', 0),
                                             ('last', 0)])
def test_tc_neighbour_tables(pattern, density, enc):
    for cin, cout in [(32, 64), (128, 128)]:
        run_tc(cin, cout, ENC[enc], pattern=pattern, density=density, mask='exact', residual=True, seed=11, tag=pattern)


def test_tc_f16_output_saturates():
    """An f16 output beyond +-65504 is stored as +-65504 (include/srfdet_b200.h), never as inf."""
    bias = torch.zeros(64)
    bias[::3] = 7.0e4
    bias[1::3] = -9.0e4
    r = run_tc(64, 64, F16, F16, bias=bias, relu=False, check=False, seed=2)
    got, ref = r['got'], r['ref']
    assert torch.isfinite(got).all()
    hi, lo = ref > 65504, ref < -65504
    assert hi.sum() > 1000 and lo.sum() > 1000
    assert (got[hi] == 65504).all() and (got[lo] == -65504).all()
    ok = ~(hi | lo)
    check_bound(got[ok], ref[ok], r['s'][ok], F16, EPS_TC, 'saturation, in-range elements')


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('cin,cout', [(128, 128), (64, 64), (32, 16), (16, 32)])
def test_tc_dense_scatter(cin, cout, enc):
    """conv_out form: kvol 3, result scattered into a zeroed (B, cout * D, H, W) f32 map, batch 2, D = 2.  Cells no row
    visits and the cells of rows past the count must stay 0."""
    _dense_case('tc', cin, cout, ENC[enc])


def _dense_case(kind, cin, cout, enc, relu=True, residual=False):
    L, lib = _lib()
    B, D, H, W = 2, 2, 20, 24
    cap, n_in, kvol = 512, 2000, 3
    g = torch.Generator().manual_seed(cin + cout + enc)
    cells = torch.randperm(B * D * H * W, generator=g)[:cap]
    coors = torch.stack([cells // (D * H * W), (cells // (H * W)) % D, (cells // W) % H, cells % W], 1).to(torch.int32)
    live = cap - 77
    x = torch.randn(n_in, cin, generator=g).cuda()
    w = (torch.randn(kvol, cin, cout, generator=g) / (kvol * cin / 3) ** 0.5).cuda()
    bias = (torch.randn(cout, generator=g) * 0.5).cuda()
    nbr = table('random', kvol, cap, n_in, g, 0.7).cuda()
    res = torch.randn(cap, cout, generator=g).cuda() if residual else None
    st = L.stream_ptr()
    if kind == 'tc':
        xe = _convert(x, enc)
        wp = torch.empty(L.enc_width(enc, kvol * cin * cout), dtype=L.enc_torch_dtype(enc), device='cuda')
        L.check(lib.srf_pack_weight_tc(_ptr(w), kvol, cin, cout, enc, _ptr(wp), st), 'pack')
    else:
        xe, wp = encode(x, enc), w.contiguous()
    dense = torch.zeros((B, cout * D, H, W), dtype=torch.float32, device='cuda')
    cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
    coors_d = coors.cuda().contiguous()
    a = L.ConvArgs()
    a.in_, a.in_dtype, a.in_rows, a.cin, a.cout, a.kvol = _ptr(xe), enc, n_in, cin, cout, kvol
    a.nbr, a.tile_mask, a.cap_out, a.d_n_out = _ptr(nbr), _ptr(exact_mask(nbr, live, cap)), cap, _ptr(cnt)
    a.w, a.bias, a.residual, a.relu = _ptr(wp), _ptr(bias), _ptr(res), int(relu)
    a.out, a.out_dtype, a.dense, a.out_coors = None, F32, _ptr(dense), _ptr(coors_d)
    a.out_dims[0], a.out_dims[1], a.out_dims[2], a.out_dims[3] = B, D, H, W
    fn = lib.srf_spconv_tc if kind == 'tc' else lib.srf_spconv_f32
    L.check(fn(ctypes.byref(a), st), f'{kind} dense')
    torch.cuda.synchronize()
    ref, s = reference(x, w, nbr, live, enc, bias, None if res is None else res.double(), relu,
                       w_enc=enc if kind == 'tc' else F32)
    want = torch.zeros((B, cout, D, H, W), dtype=torch.float64, device='cuda')
    bound = torch.zeros_like(want)
    eps = EPS_TC if kind == 'tc' else EPS_SIMT
    c = coors[:live].long().cuda()
    want[c[:, 0], :, c[:, 1], c[:, 2], c[:, 3]] = ref
    bound[c[:, 0], :, c[:, 1], c[:, 2], c[:, 3]] = s
    got = dense.view(B, cout, D, H, W).double()
    # unvisited cells (bound 0) must be exactly 0
    check_bound(got, want, bound, F32, eps, f'{kind} dense {cin}->{cout} enc {enc}', (kind, enc, 'dense'))


def test_tc_16_to_16_both_kernels():
    """16 -> 16 with a same-encoding output runs the warp-MMA kernel; with SRF_CONV16_WARP=0 the same call runs the
    tcgen05 G = 4 kernel.  Both are checked against the reference, in a subprocess for the tcgen05 form (the switch is
    read once per process)."""
    for enc in (F16, BF16):
        run_tc(16, 16, enc, residual=True, relu=True, seed=31)
    code = ('import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n'
            'import test_gpu_spconv as t\n'
            'for e in (t.F16, t.BF16):\n'
            '    t.run_tc(16, 16, e, residual=True, relu=True, seed=31)\n'
            'print("ok")\n') % (os.path.dirname(os.path.abspath(__file__)), os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    with tempfile.TemporaryDirectory() as d:
        p = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, SRF_CONV16_WARP='0'), cwd=d,
                           capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and 'ok' in p.stdout, p.stdout + p.stderr


# ------------------------------------------------------------------------------------------------ srf_spconv_f32 (SIMT)
def run_simt(cin, cout, in_enc, out_enc=F32, kvol=27, cap=512, n_in=1500, mask='none', residual=False, relu=True,
             seed=0, nbr=None, tag=''):
    L, lib = _lib()
    g = torch.Generator().manual_seed(seed)
    live = cap - 29
    x = torch.randn(n_in, cin, generator=g).cuda()
    w = (torch.randn(kvol, cin, cout, generator=g) / (kvol * cin / 3) ** 0.5).cuda()
    bias = (torch.randn(cout, generator=g) * 0.5).cuda()
    if nbr is None:
        nbr = table('random', kvol, cap, n_in, g, 0.5)
    nbr = nbr.cuda().contiguous()
    res_t = encode(torch.randn(cap, cout, generator=g).cuda(), out_enc) if residual else None
    if isinstance(mask, torch.Tensor):
        tm = mask.cuda()
    else:
        tm = {'none': None, 'exact': exact_mask(nbr, live, cap),
              'ones': torch.full((cap // 128,), -1, dtype=torch.int32, device='cuda')}[mask]
    xe = encode(x, in_enc)
    cnt = torch.tensor([live], dtype=torch.int32, device='cuda')
    out = torch.empty((cap, L.enc_width(out_enc, cout)), dtype=L.enc_torch_dtype(out_enc), device='cuda')
    out.view(torch.int16 if out.dtype != torch.float32 else torch.int32).fill_(0x3F1B)
    sentinel = out.clone()
    a = L.ConvArgs()
    a.in_, a.in_dtype, a.in_rows, a.cin, a.cout, a.kvol = _ptr(xe), in_enc, n_in, cin, cout, kvol
    a.nbr, a.tile_mask, a.cap_out, a.d_n_out = _ptr(nbr), _ptr(tm), cap, _ptr(cnt)
    a.w, a.bias, a.residual, a.relu, a.out, a.out_dtype = _ptr(w), _ptr(bias), _ptr(res_t), int(relu), _ptr(out), out_enc
    L.check(lib.srf_spconv_f32(ctypes.byref(a), L.stream_ptr()), f'srf_spconv_f32 {tag}')
    torch.cuda.synchronize()
    ref, s = reference(x, w, nbr, live, in_enc, bias, decode(res_t, cout) if residual else None, relu, w_enc=F32)
    check_bound(decode(out[:live], cout), ref, s, out_enc, EPS_SIMT, f'simt {cin}->{cout} in {in_enc} out {out_enc} {tag}',
                ('simt', in_enc, out_enc))
    assert torch.equal(out[live:], sentinel[live:]), 'rows past the count were written'


@pytest.mark.parametrize('in_enc', ['f32', 'bf16'])
@pytest.mark.parametrize('cout', [16, 32, 64, 128])
@pytest.mark.parametrize('cin', [1, 3, 4, 5, 8, 16, 24, 64, 128])
def test_simt_channels(cin, cout, in_enc):
    """Small-cin kernel (f32 in, cin <= 8, cout 16 / 32, no residual) and the general kernel; a residual forces the latter."""
    run_simt(cin, cout, ENC[in_enc], seed=cin * 3 + cout)
    run_simt(cin, cout, ENC[in_enc], residual=True, relu=False, seed=cin * 3 + cout + 1, tag='residual')


@pytest.mark.parametrize('out', ['f32', 'bf16', 'f16', 'bf16x2', 'f16x2'])
@pytest.mark.parametrize('cin,cout', [(4, 16), (5, 32), (16, 64), (128, 128)])
def test_simt_output_encodings(cin, cout, out):
    for residual in (False, True):
        run_simt(cin, cout, F32, ENC[out], residual=residual, seed=cout + residual, tag='out enc')


@pytest.mark.parametrize('mask', ['none', 'exact', 'ones', 'empty'])
@pytest.mark.parametrize('cin,cout,in_enc', [(4, 16, F32), (5, 32, F32), (32, 64, BF16), (64, 128, F32)])
def test_simt_tile_masks(cin, cout, in_enc, mask):
    cap, n_in = 1024, 1500
    g = torch.Generator().manual_seed(41)
    nbr = table('random', 27, cap, n_in, g, 0.5)
    if mask == 'empty':
        nbr.view(27, cap // 128, 128)[:, 2::3] = -1
        m = exact_mask(nbr.cuda(), cap - 29, cap)
    else:
        m = mask
    run_simt(cin, cout, in_enc, cap=cap, n_in=n_in, nbr=nbr, mask=m, seed=9, tag=mask)
    run_simt(cin, cout, in_enc, cap=cap, n_in=n_in, nbr=nbr, mask=m, residual=True, seed=9, tag=mask + ' residual')


@pytest.mark.parametrize('cin,cout,in_enc', [(4, 16, F32), (64, 128, F32), (16, 32, BF16)])
def test_simt_dense_scatter(cin, cout, in_enc):
    _dense_case('simt', cin, cout, in_enc, residual=False)
    _dense_case('simt', cin, cout, in_enc, relu=False, residual=True)


# ------------------------------------------------------------------------------------------------ dense-rulebook path
def dense_rulebook_np(n, h, w, ks, stride, pad, cap):
    ho, wo = (h + 2 * pad - ks) // stride + 1, (w + 2 * pad - ks) // stride + 1
    nbr = np.full((ks * ks, cap), -1, np.int32)
    rows = np.arange(n * ho * wo)
    ox, oy, img = rows % wo, (rows // wo) % ho, rows // (wo * ho)
    for k in range(ks * ks):
        iy, ix = oy * stride - pad + k // ks, ox * stride - pad + k % ks
        ok = (iy >= 0) & (iy < h) & (ix >= 0) & (ix < w)
        nbr[k, rows[ok]] = ((img * h + iy) * w + ix)[ok]
    return nbr, ho, wo


@pytest.mark.parametrize('h,w', [(23, 37), (5, 3)])
@pytest.mark.parametrize('stride', [1, 2])
def test_dense_rulebook_tables(h, w, stride):
    """srf_dense_rulebook == the numpy construction bit for bit; its tile masks cover the exact masks (the builder sets
    every kvol bit of a live tile) and are 0 on tiles past n*ho*wo."""
    L, lib = _lib()
    n, ks, pad = 2, 3, 1
    ho, wo = (h + 2 * pad - ks) // stride + 1, (w + 2 * pad - ks) // stride + 1
    cap = -(-n * ho * wo // 128) * 128 + 128
    want, _, _ = dense_rulebook_np(n, h, w, ks, stride, pad, cap)
    nbr = torch.full((ks * ks, cap), -7, dtype=torch.int32, device='cuda')
    tm = torch.full((cap // 128,), -7, dtype=torch.int32, device='cuda')
    L.check(lib.srf_dense_rulebook(n, h, w, ks, stride, pad, cap, _ptr(nbr), _ptr(tm), L.stream_ptr()), 'rulebook')
    torch.cuda.synchronize()
    assert np.array_equal(nbr.cpu().numpy(), want)
    ex = exact_mask(nbr, n * ho * wo, cap).cpu().numpy().view(np.uint32)
    got = tm.cpu().numpy().view(np.uint32)
    assert ((got & ex) == ex).all()
    live = np.arange(cap // 128) * 128 < n * ho * wo
    assert (got[live] == (1 << ks * ks) - 1).all() and (got[~live] == 0).all()


@pytest.mark.parametrize('enc', ENCS)
@pytest.mark.parametrize('cin,cout', [(64, 64), (64, 128), (128, 256)])
@pytest.mark.parametrize('h,w,stride', [(23, 37, 1), (23, 37, 2), (5, 3, 1), (5, 3, 2)])
def test_dense_rulebook_conv_vs_conv2d(h, w, stride, cin, cout, enc):
    """srf_spconv_tc over srf_dense_rulebook tables (the SECONDCustom path) == float64 conv2d of the used operands."""
    L, lib = _lib()
    e = ENC[enc]
    n, ks, pad = 2, 3, 1
    ho, wo = (h + 2 * pad - ks) // stride + 1, (w + 2 * pad - ks) // stride + 1
    cap = -(-n * ho * wo // 128) * 128
    g = torch.Generator().manual_seed(h * stride + cin)
    img = torch.randn(n, cin, h, w, generator=g).cuda()
    wt = (torch.randn(cout, cin, ks, ks, generator=g) / (9 * cin / 3) ** 0.5).cuda()
    bias = (torch.randn(cout, generator=g) * 0.5).cuda()
    rows = img.permute(0, 2, 3, 1).reshape(n * h * w, cin).contiguous()
    w_kio = wt.permute(2, 3, 1, 0).reshape(ks * ks, cin, cout).contiguous()        # k = ky * ks + kx
    nbr = torch.empty((ks * ks, cap), dtype=torch.int32, device='cuda')
    tm = torch.empty((cap // 128,), dtype=torch.int32, device='cuda')
    st = L.stream_ptr()
    L.check(lib.srf_dense_rulebook(n, h, w, ks, stride, pad, cap, _ptr(nbr), _ptr(tm), st), 'rulebook')
    xe = _convert(rows, e)
    wp = torch.empty(L.enc_width(e, ks * ks * cin * cout), dtype=L.enc_torch_dtype(e), device='cuda')
    L.check(lib.srf_pack_weight_tc(_ptr(w_kio), ks * ks, cin, cout, e, _ptr(wp), st), 'pack')
    out = torch.empty((cap, L.enc_width(F32, cout)), dtype=torch.float32, device='cuda')
    a = L.ConvArgs()
    a.in_, a.in_dtype, a.in_rows, a.cin, a.cout, a.kvol = _ptr(xe), e, n * h * w, cin, cout, ks * ks
    a.nbr, a.tile_mask, a.cap_out, a.d_n_out = _ptr(nbr), _ptr(tm), cap, None
    a.w, a.bias, a.residual, a.relu, a.out, a.out_dtype = _ptr(wp), _ptr(bias), None, 1, _ptr(out), F32
    L.check(lib.srf_spconv_tc(ctypes.byref(a), st), 'conv')
    torch.cuda.synchronize()
    xh, xl = (t.double() for t in split_parts(img, e))
    wh, wl = (t.double() for t in split_parts(wt, e))
    conv = lambda u, v: torch.nn.functional.conv2d(u, v, stride=stride, padding=pad)
    ref = conv(xh, wh) + (conv(xl, wh) + conv(xh, wl) if e in SPLIT else 0) + bias.double()[None, :, None, None]
    s = conv(xh.abs(), wh.abs()) + bias.double().abs()[None, :, None, None]
    ref = torch.relu(ref).permute(0, 2, 3, 1).reshape(-1, cout)
    s = s.permute(0, 2, 3, 1).reshape(-1, cout)
    check_bound(out[:n * ho * wo].double(), ref, s, F32, EPS_TC, f'dense rulebook {h}x{w}/{stride} {cin}->{cout} {enc}',
                ('tc', e, F32))


# ------------------------------------------------------------------------------------------------ srf_convert_rows
@pytest.mark.parametrize('enc', ['bf16', 'f16', 'bf16x2', 'f16x2'])
def test_convert_rows_bit_exact(enc):
    """srf_convert_rows == torch rounding bit for bit: c_pad > c zero padded, f16 subnormals, saturation at +-65504."""
    L, lib = _lib()
    e = ENC[enc]
    g = torch.Generator().manual_seed(5)
    rows, c, c_pad = 777, 37, 48
    v = torch.randn(rows, c, generator=g) * torch.exp2(torch.randint(-30, 18, (rows, c), generator=g).float())
    v[0, :8] = torch.tensor([65504.0, -65504.0, 65519.0, 65520.0, 1.0e5, -3.0e5, 6.0e-8, -2.9e-8])
    v[1, :6] = torch.tensor([2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -26, 6.1e-5, -5.9e-5, 0.0])
    v = v.cuda()
    out = torch.empty((rows, L.enc_width(e, c_pad)), dtype=L.enc_torch_dtype(e), device='cuda')
    out.fill_(1.0)
    L.check(lib.srf_convert_rows(_ptr(v), rows, c, c_pad, e, _ptr(out), L.stream_ptr()), 'convert')
    torch.cuda.synchronize()
    hi, lo = split_parts(v, e)
    pad = torch.zeros(rows, c_pad - c, device='cuda')
    want = torch.cat([hi, pad] + ([lo, pad] if e in SPLIT else []), 1).to(out.dtype)
    assert torch.equal(out.view(torch.int16), want.view(torch.int16))
    if is_f16(e):
        assert torch.isfinite(out.float()).all()
        assert (out[:, :c].float().abs() < 2.0 ** -14).logical_and(out[:, :c].float() != 0).any()   # subnormals produced


# ------------------------------------------------------------------------------------------------ argument checks
def test_argument_checks_do_not_launch():
    """Rejected calls return their error code before any launch (the launch counter does not move)."""
    L, lib = _lib()
    cap = 256
    buf = torch.zeros(1 << 16, dtype=torch.float32, device='cuda')
    nbr = torch.full((27, cap), -1, dtype=torch.int32, device='cuda')
    coors = torch.zeros((cap, 4), dtype=torch.int32, device='cuda')

    def args(**kw):
        a = L.ConvArgs()
        a.in_, a.in_dtype, a.in_rows, a.cin, a.cout, a.kvol = _ptr(buf), F16, 64, 32, 32, 27
        a.nbr, a.tile_mask, a.cap_out, a.d_n_out = _ptr(nbr), None, cap, None
        a.w, a.bias, a.residual, a.relu, a.out, a.out_dtype = _ptr(buf), None, None, 0, _ptr(buf), F16
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    cases = [(lib.srf_spconv_tc, args(cin=48), ERR_UNSUPPORTED),
             (lib.srf_spconv_tc, args(cin=64, cout=48), ERR_UNSUPPORTED),
             (lib.srf_spconv_tc, args(cap_out=200), ERR_ARG),
             (lib.srf_spconv_tc, args(cout=256, out=None, out_dtype=F32, dense=_ptr(buf), out_coors=_ptr(coors)), ERR_ARG),
             (lib.srf_spconv_tc, args(kvol=0), ERR_ARG),
             (lib.srf_spconv_tc, args(kvol=28), ERR_ARG),
             (lib.srf_spconv_tc, args(in_dtype=F32), ERR_ARG),
             (lib.srf_spconv_tc, args(out_dtype=BF16), ERR_ARG),
             (lib.srf_spconv_f32, args(in_dtype=F16), ERR_ARG),
             (lib.srf_spconv_f32, args(in_dtype=F16X2), ERR_ARG),
             (lib.srf_spconv_f32, args(in_dtype=BF16X2), ERR_ARG),
             (lib.srf_spconv_f32, args(in_dtype=F32, kvol=28), ERR_ARG),
             (lib.srf_spconv_f32, args(in_dtype=F32, cap_out=200), ERR_ARG)]
    torch.cuda.synchronize()
    n0 = lib.srf_launch_count()
    for i, (fn, a, rc) in enumerate(cases):
        assert fn(ctypes.byref(a), L.stream_ptr()) == rc, (i, lib.srf_last_error())
    assert lib.srf_launch_count() == n0


@pytest.fixture(scope='module', autouse=True)
def _report_ratios():
    """Largest bound ratio per (kernel, in encoding, out encoding) of this run: the EPS_* calibration.  Printed, and
    written as JSON to the file SRF_SPCONV_RATIOS names, if set."""
    yield
    import json
    rows = {f'{k}/{i}/{o}': v for (k, i, o), v in sorted(_ratios.items(), key=str)}
    print('\nbound ratios:', json.dumps(rows, indent=1))
    path = os.environ.get('SRF_SPCONV_RATIOS')
    if path:
        with open(path, 'w') as f:
            json.dump(rows, f, indent=1)
