"""Per-entry-point CUDA-event timing of the C-ABI calls (bench.py's per-kernel-family rooflines).

`capture()` wraps every function of the loaded library so that each call is bracketed by two CUDA
events on the stream it is enqueued on and its integer arguments are recorded; `families()` groups
the calls and attaches the ALGORITHMIC work of each (SURVEY.md 8d: compulsory bytes and flops,
not the traffic the implementation happens to generate).  Used only for measurement: the wrappers
are installed on demand and removed afterwards, the product path calls the bare functions.
"""
import contextlib

import torch

from . import _lib as L

ES = {L.F32: 4, L.BF16: 2, L.F16: 2, L.BF16X2: 4, L.F16X2: 4}      # bytes per value of an encoding


def _iv(x):
    """ctypes argument -> python int when it is one, tuple of ints for a small host array (dims, kernel sizes)."""
    try:
        return int(x)
    except (TypeError, ValueError):
        pass
    try:
        if 0 < len(x) <= 8:
            return tuple(int(v) for v in x)
    except (TypeError, ValueError):
        pass
    return None


class Capture:
    def __init__(self):
        self.calls = []       # (name, args tuple, struct summary, start event, end event)
        self.per_call = []    # (ms, name, family) filled by families()


@contextlib.contextmanager
def capture():
    lib = L.load()
    cap = Capture()
    originals = {}
    for name in L.PROTOTYPES:
        fn = getattr(lib, name)
        originals[name] = fn
        if name.endswith(('_bytes', '_splits', '_splits_enc', '_tile_k', '_tile_n', '_tile_k_enc')) or name in (
                'srf_version', 'srf_last_error', 'srf_sm_count', 'srf_launch_count', 'srf_geom_init', 'srf_conv3x3_last_used_tma'):
            continue

        def wrapped(*args, _fn=fn, _name=name):
            summary = None
            a0 = getattr(args[0], '_obj', None) if args else None
            if isinstance(a0, L.ConvArgs):
                summary = dict(cin=a0.cin, cout=a0.cout, kvol=a0.kvol, cap=a0.cap_out, in_enc=a0.in_dtype, out_enc=a0.out_dtype,
                               dense=bool(a0.dense), in_rows=a0.in_rows)
            elif isinstance(a0, L.LinearArgs):
                summary = dict(enc=a0.a_enc, m=a0.m, k=a0.k, n=a0.n, out_enc=a0.out_enc, out2=bool(a0.out2), out2_enc=a0.out2_enc,
                               k_splits=max(1, a0.k_splits))
            elif isinstance(a0, L.Map):
                a1 = getattr(args[1], '_obj', None)
                summary = dict(ca=a0.c, cb=a1.c if isinstance(a1, L.Map) and a1.ptr else 0)
            elif isinstance(a0, L.Pyramid):
                summary = dict(channels=a0.channels, levels=a0.n_levels, hw=[(a0.h[i], a0.w[i]) for i in range(a0.n_levels)])
                for a in args:
                    o = getattr(a, '_obj', None)
                    if isinstance(o, L.RoiOut):
                        summary['out_enc'] = o.dtype
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = _fn(*args)
            e1.record()
            cap.calls.append((_name, tuple(_iv(a) for a in args), summary, e0, e1))
            return rc
        setattr(lib, name, wrapped)
    try:
        yield cap
    finally:
        for name, fn in originals.items():
            setattr(lib, name, fn)


def _family(name, a, s):
    if name in ('srf_hard_voxelize', 'srf_dynamic_voxelize'):
        return 'voxelize'
    if name in ('srf_dynamic_vfe', 'srf_dynamic_scatter'):
        return 'dynamic VFE'
    if name == 'srf_rulebook_build':
        return 'rulebook build'
    if name in ('srf_index_clear', 'srf_index_finalize'):
        return 'cell index: clear + rank scan'
    if name.startswith('srf_index_') or name == 'srf_gather_rows':
        return 'cell index: mark / emit / lookup'
    if name in ('srf_spconv_tc', 'srf_spconv_f32', 'srf_spconv_bf16'):
        if s['kvol'] == 9:
            return f"dense conv3x3 {s['cin']}->{s['cout']}"
        return f"sparse conv {s['cin']}->{s['cout']}" + (' (first layer, FFMA)' if name == 'srf_spconv_f32' else '')
    if name == 'srf_conv3x3_rows':
        return f'dense conv3x3 {a[5]}->{a[7]}'
    if name == 'srf_bev_roi_features':
        return 'BEV RoIAlign'
    if name == 'srf_img_roi_features':
        return 'image RoIAlign (6 cameras)'
    if name in ('srf_linear', 'srf_linear_tc', 'srf_linear_bf16'):
        m, k, n = (s['m'], s['k'], s['n']) if name == 'srf_linear' else ((a[2], a[3], a[5]) if name == 'srf_linear_tc' else (a[1], a[2], a[4]))
        return f'GEMM {k}->{n}' + (' (pixel rows)' if m > 5000 and k <= 512 and m != 44100 else '')
    if name in ('srf_linear_f32', 'srf_gemv_f32'):
        return 'small projections (FFMA)'
    if name.startswith('srf_dynconv_interact'):
        return 'DynamicConv interaction'
    if name.startswith('srf_layernorm'):
        return 'LayerNorm (split-K reduce / residual)'
    if name == 'srf_mha_attention':
        return 'self-attention core'
    if name in ('srf_dwconv3x3_s2', 'srf_channel_sum', 'srf_dpg_mix'):
        return 'DPG staircase'
    if name in ('srf_convert_rows', 'srf_nchw_to_rows', 'srf_upsample_add', 'srf_f32_to_bf16'):
        return 'layout / encoding passes'
    if name in ('srf_apply_deltas', 'srf_decode_boxes', 'srf_boxes_to_corners'):
        return 'box update / decode'
    if name.startswith('srf_pack') or name == 'srf_dense_rulebook':
        return None            # one-time weight packing / static tables: not part of a frame
    return 'other'


def _work(name, a, s, ctx):
    """(flops, bytes) of one call: algorithmic work."""
    n_pts, c_pts = ctx['n_points'], ctx['c_points']
    if name == 'srf_hard_voxelize':
        m = ctx['n_voxels']
        return 0.0, n_pts * c_pts * 4 + m * (16 + 4) + m * c_pts * 4
    if name == 'srf_dynamic_voxelize':
        return 0.0, n_pts * c_pts * 4 + n_pts * 16
    if name in ('srf_dynamic_vfe', 'srf_dynamic_scatter'):
        return 0.0, 3 * (n_pts * c_pts * 4 + n_pts * 4 + ctx['n_voxels'] * c_pts * 4) + n_pts * (c_pts + 35) * 4
    if name in ('srf_spconv_tc', 'srf_spconv_f32', 'srf_spconv_bf16'):
        return None            # filled from the rulebooks (sparse) / the grid (dense) by the caller
    if name == 'srf_conv3x3_rows':
        rows, cin, cout = a[2] * a[3] * a[4], a[5], a[7]
        return 2.0 * rows * 9 * cin * cout, rows * cin * ES[a[1]] + rows * cout * ES[a[11]] + 9 * cin * cout * ES[a[1]]
    if name == 'srf_bev_roi_features':
        c = s['channels']
        k = a[2] * a[3]
        return 0.0, k * 49 * c * ES[s.get('out_enc', L.F32)] + sum(h * w for h, w in s['hw']) * c * 4
    if name == 'srf_img_roi_features':
        # output + the part of the 6-camera pyramid the proposals actually touch.  SURVEY 8d gives the whole pyramid
        # (379 MB) as an upper bound; what 900 car-sized proposals touch is data dependent and ~6x smaller: the
        # per-launch DRAM read of this kernel in the committed ncu capture is used when bench.py passes it
        # (ctx['img_roi_input_bytes']), otherwise the upper bound.
        # (a batch of B samples touches B such camera sets)
        c = s['channels']
        batch, k, n_cam = a[2], a[2] * a[3], a[6]
        touched = batch * (ctx.get('img_roi_input_bytes') or n_cam * sum(h * w for h, w in s['hw']) * c * 4)
        return 0.0, k * 49 * c * ES[s.get('out_enc', L.F32)] + touched
    if name == 'srf_linear':
        es = ES[s['enc']]
        return 2.0 * s['m'] * s['k'] * s['n'], s['m'] * s['k'] * es + s['k'] * s['n'] * es + s['m'] * s['n'] * (
            ES[s['out_enc']] * s['k_splits'] + (ES[s['out2_enc']] if s['out2'] else 0))
    if name == 'srf_linear_tc':
        enc, m, k, n, out_enc = a[1], a[2], a[3], a[5], a[13]
        return 2.0 * m * k * n, m * k * ES[enc] + k * n * ES[enc] + m * n * ES[out_enc] * max(1, a[14] or 1)
    if name == 'srf_linear_f32' or name == 'srf_gemv_f32':
        m, k, n = a[1], a[2], a[4]
        return 2.0 * m * k * n, (m * k + k * n + m * n) * 4
    if name == 'srf_dynconv_interact_tc':
        k, c, d = a[4], a[5], a[6]
        return 2.0 * k * 49 * c * d * 2, k * 49 * c * ES[a[1]] + k * 2 * c * d * ES[a[3]] + k * 49 * c * ES[a[14]]
    if name == 'srf_layernorm_enc':
        rows, n, parts = a[2], a[3], a[4]
        return 0.0, rows * n * 4 * (parts + 1)
    if name == 'srf_mha_attention':
        b, p, h, hd = a[1], a[2], a[3], a[4]
        return 4.0 * b * p * p * h * hd, b * p * h * hd * 4 * 4
    # ---- geometry (cell index + rulebook): bytes of the bitmap / rank words, coordinates and tables that MUST move
    counts = ctx.get('level_counts', {})

    def cells(d):
        return d[0] * d[1] * d[2] * d[3]

    def n_of(d, cap):
        return min(counts.get(tuple(d), cap), cap)
    if name == 'srf_index_clear':
        return 0.0, a[1] / 8                                       # bitmap written
    if name == 'srf_index_finalize':
        return 0.0, a[1] / 8 * 2                                   # bitmap read, per-word ranks written
    if name == 'srf_index_mark':
        n = n_of(a[1], a[3])
        return 0.0, n * (16 + 4)                                   # coordinates read, one bitmap word touched per voxel
    if name == 'srf_index_mark_strided':
        return 0.0, min(ctx.get('n_voxels', a[3]), a[3]) * 16 + cells(a[1]) / 8     # input coordinates read, output bitmap touched
    if name == 'srf_index_emit_coors':
        return 0.0, cells(a[1]) / 8 * 2 + n_of(a[1], a[3]) * 16    # bitmap + ranks read, coordinates written
    if name in ('srf_index_perm', 'srf_index_lookup'):
        return 0.0, a[3] * (16 + 8 + 4)
    if name == 'srf_gather_rows':
        return 0.0, a[3] * a[4] * 4 * 2 + a[3] * 4
    if name == 'srf_rulebook_build':
        kvol = a[6][0] * a[6][1] * a[6][2]
        n = min(ctx.get('cap_counts', {}).get(a[4], a[4]), a[4])
        return 0.0, n * 16 + kvol * n * 4 + cells(a[1]) / 8 * 2    # out coordinates, the table, the probed index once
    # ---- DPG staircase (fp32 maps read once, result written)
    if name == 'srf_dwconv3x3_s2':
        n, h, w = a[2], a[3], a[4]
        c = s['ca'] + s['cb']
        ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
        return 2.0 * 9 * n * ho * wo * c, (n * h * w * c + n * ho * wo * c) * 4
    if name == 'srf_channel_sum':
        n_s, group, h, w = a[2], a[3], a[4], a[5]
        return 0.0, n_s * group * h * w * (s['ca'] + s['cb']) * 4
    if name == 'srf_dpg_mix':
        return 0.0, a[2] * a[3] * a[4] * 4 * 2 + a[3] * a[4] * (a[6] + a[8]) * 4
    # ---- layout / encoding passes
    if name == 'srf_convert_rows':
        return 0.0, a[1] * a[2] * 4 + a[1] * a[3] * ES[a[4]]
    if name == 'srf_nchw_to_rows':
        return 0.0, a[1] * a[2] * a[3] * a[4] * (4 + ES[a[5]])
    if name == 'srf_upsample_add':
        return 0.0, a[2] * a[3] * a[4] * a[7] * ES[a[8]] * 2 + a[2] * a[5] * a[6] * a[7] * ES[a[8]]
    if name == 'srf_apply_deltas':
        return 0.0, a[2] * a[3] * 4 * 3
    if name == 'srf_decode_boxes':
        return 0.0, (a[1] * 2 + a[3] * a[4] * 2) * 4
    return 0.0, 0.0


def families(cap, ctx, peaks):
    """Group the captured calls of ONE frame -> list of dicts (family, launches, ms, flops, bytes, bound, achieved, frac)."""
    torch.cuda.synchronize()
    groups = {}
    for name, a, s, e0, e1 in cap.calls:
        fam = _family(name, a, s)
        if fam is None:
            continue
        ms = e0.elapsed_time(e1)
        w = _work(name, a, s, ctx)
        if w is None:
            w = ctx['conv_work'](s)
        cap.per_call.append((round(ms, 4), name, fam))
        g = groups.setdefault(fam, dict(family=fam, launches=0, ms=0.0, flops=0.0, bytes=0.0, entry_points=set()))
        g['launches'] += 1
        g['ms'] += ms
        g['flops'] += w[0]
        g['bytes'] += w[1]
        g['entry_points'].add(name)
    ridge = peaks['tf_sust'] * 1e12 / (peaks['hbm'] * 1e9)
    out = []
    for g in groups.values():
        g['entry_points'] = sorted(g['entry_points'])
        t = g['ms'] * 1e-3
        gbs = g['bytes'] / t / 1e9 if t > 0 else 0.0
        tfs = g['flops'] / t / 1e12 if t > 0 else 0.0
        tensor = g['bytes'] > 0 and g['flops'] / g['bytes'] >= ridge
        g.update(ms=round(g['ms'], 4), bound='tensor' if tensor else 'hbm', achieved=round(tfs if tensor else gbs, 2),
                 unit='TFLOP/s' if tensor else 'GB/s', peak=peaks['tf_sust'] if tensor else peaks['hbm'],
                 frac=round((tfs / peaks['tf_sust']) if tensor else (gbs / peaks['hbm']), 4),
                 gbs=round(gbs, 1), tflops=round(tfs, 2))
        out.append(g)
    out.sort(key=lambda g: -g['ms'])
    return out
