"""Sparse-region-fusion head stages under the reference names
(mmdet3d_plugin/models/sparse_heads/srfdet_head.py): DynamicConv (:2633-2693),
SingleSRFDetHeadLiDAR (:1348-1623) and SingleSRFDetHead (:2103-2629).

Hot path (SURVEY.md 8 rows a6-a10) on the CUDA kernels of this package: RoI sampling,
fusion projection, DynamicConv.  The remaining dense rows of a stage (self-attention over
the proposals, FFN, cls/reg towers, apply_deltas; SURVEY 8f rank 2) run as plain torch ops
so the five stages chain with real boxes; they are not part of the measured path.
Parameter names equal the reference's, so its checkpoints load unchanged.
"""
import ctypes
import math

import torch
import torch.nn.functional as F
from torch import nn

from .. import _lib as L
from . import registry
from .registry import HEADS
from .roi import flat_image_maps, img_feats_sampling_bboxes_roi, maps_channels_last, points_feats_sampling_bboxes_roi

_DEFAULT_SCALE_CLAMP = math.log(100000.0 / 16)


def _f(t):
    return t.detach().float().contiguous()


class _LinearView:
    """(weight (n,k), bias) pair with nn.Linear's attribute names (MultiheadAttention.in_proj_*, folded 1x1 convs)."""

    def __init__(self, weight, bias):
        self.weight, self.bias = weight, bias
        self.out_features, self.in_features = weight.shape


def _cached(cache, key, src, make):
    """Packed / folded form of `src` tensors, rebuilt when any of them was replaced or written
    in place (load_state_dict at any level of the module tree, optimizer step, manual edit)."""
    ver = tuple((t.data_ptr(), t._version) for t in src)
    hit = cache.get(key)
    if hit is None or hit[0] != ver:
        hit = (ver, make())
        cache[key] = hit
    return hit[1]


def _encode_out(x, enc):
    return x if enc == L.F32 else encode_rows(x, enc)


def encode_rows(x, enc):
    """(M,K) fp32 -> (M, K | 2K) tensor in the 16-bit encoding `enc` (srf_convert_rows)."""
    m, k = x.shape
    out = torch.empty((m, L.enc_width(enc, k)), dtype=L.enc_torch_dtype(enc), device=x.device)
    L.check(L.load().srf_convert_rows(L.ptr(_f(x)), m, k, k, enc, L.ptr(out), L.stream_ptr()), 'srf_convert_rows')
    return out


def _linear(x, lin, precision, cache, key, relu=False, ln=None, out_enc=None, residual=None, out2_enc=None, a_cols=None,
            ln_per_tile=False):
    """nn.Linear (+LayerNorm +ReLU) on the library's GEMMs.

    x: (M,K) fp32, or an (M, K|2K) tensor already in the activation encoding of `precision`.
    'fp32_simt': FFMA kernel, fp32 in/out.  Tensor-core modes: tcgen05 GEMM on operands in the
    mode's encoding (weights packed once, re-packed when they change); the result is written in
    `out_enc` (default: the mode's activation encoding; L.F32 for an fp32 result).
    residual (M,N) fp32: added before the LayerNorm.  out2_enc: additionally return a second copy of the
    result in that encoding (-> (out, out2)).  a_cols=(c0, width): A is the column block [c0, c0+K) of an encoded
    buffer whose rows have `width` logical columns.  ln_per_tile: `ln` holds N parameters and every 128-column tile is
    normalised on its own (two towers merged into one GEMM)."""
    lib = L.load()
    m = x.shape[0]
    k, n = lin.in_features, lin.out_features
    dev = x.device
    st = L.stream_ptr()
    bias = _f(lin.bias) if lin.bias is not None else None
    enc = registry.act_enc(precision)
    if enc is not None:
        # shapes the tcgen05 tiles cannot cover (not multiples of 16, or of the tile above it) take the FFMA kernel
        tk = lib.srf_linear_tile_k_enc(k, enc)
        if min(k, tk) not in (16, 32, 64, 128) or min(n, 128) not in (16, 32, 64, 128) or k % tk or (n > 128 and n % 128) \
                or (ln is not None and n > 1024):
            assert a_cols is None and not ln_per_tile
            out = _linear(L.decode(x, k) if x.dtype != torch.float32 else x, lin, 'fp32_simt', cache, key, relu, ln, residual=residual)
            res = _encode_out(out, enc if out_enc is None else out_enc)
            return (res, _encode_out(out, out2_enc)) if out2_enc is not None else res
    if enc is None:
        assert a_cols is None and not ln_per_tile
        x = _f(x)
        w = _f(lin.weight)
        out = torch.empty((m, n), dtype=torch.float32, device=dev)
        fuse_relu = relu and ln is None and residual is None
        L.check(lib.srf_linear_f32(L.ptr(x), m, k, L.ptr(w), n, L.ptr(bias), int(fuse_relu), L.ptr(out), st), 'srf_linear_f32')
        if ln is not None:
            L.check(lib.srf_layernorm_enc(L.ptr(out), L.F32, m, n, 1, None, L.ptr(residual), L.ptr(_f(ln.weight)), L.ptr(_f(ln.bias)),
                                          ln.eps, int(relu), L.ptr(out), L.F32, None, 0, st), 'srf_layernorm')
        elif residual is not None:
            out = out + residual
            out = torch.relu_(out) if relu else out
        return (out, out) if out2_enc is not None else out
    a = L.LinearArgs()
    if a_cols is not None:
        c0, width = a_cols
        assert x.dtype == L.enc_torch_dtype(enc) and x.shape[1] == L.enc_width(enc, width) and x.is_contiguous()
        a.a = x.data_ptr() + c0 * x.element_size()
        a.a_stride, a.a_lo_off = x.shape[1], width
    else:
        if x.dtype == torch.float32:
            x = encode_rows(x, enc)
        assert x.dtype == L.enc_torch_dtype(enc) and x.shape[1] == L.enc_width(enc, k), 'operand is not in the mode\'s encoding'
        x = x.contiguous()
        a.a = x.data_ptr()

    def pack():
        wp = torch.empty((L.enc_width(enc, n * k),), dtype=L.enc_torch_dtype(enc), device=dev)
        L.check(lib.srf_pack_linear_tc(L.ptr(_f(lin.weight)), n, k, enc, L.ptr(wp), st), 'srf_pack_linear_tc')
        return wp
    wp = _cached(cache, (key, enc), (lin.weight,), pack)
    out_enc = enc if out_enc is None else out_enc
    eps = float(ln.eps) if ln is not None else 1e-5

    def alloc(e):
        return torch.empty((m, L.enc_width(e, n)), dtype=L.enc_torch_dtype(e), device=dev)
    a.a_enc, a.m, a.k, a.w, a.n = enc, m, k, L.ptr(wp), n
    a.ln_eps, a.k_splits = eps, 1
    # few output tiles but a long reduction (DynamicConv.out_layer: 900 x 6272 -> 128): split K
    # over CTAs, fp32 partials in per-split slabs, bias + LayerNorm + ReLU in one pass after
    tiles = ((m + 127) // 128) * ((n + 127) // 128)
    kvol = k // lib.srf_linear_tile_k_enc(k, enc)
    if ln is not None and not ln_per_tile and tiles * 4 <= 148 and kvol >= 8:
        splits = lib.srf_linear_splits_enc(k, enc, min(kvol, max(1, 148 // tiles)))
        part = torch.empty((splits, m, n), dtype=torch.float32, device=dev)
        a.out, a.out_enc, a.k_splits = L.ptr(part), L.F32, splits
        L.check(lib.srf_linear(ctypes.byref(a), st), 'srf_linear')
        out = alloc(out_enc)
        out2 = alloc(out2_enc) if out2_enc is not None else None
        L.check(lib.srf_layernorm_enc(L.ptr(part), L.F32, m, n, splits, L.ptr(bias), L.ptr(residual), L.ptr(_f(ln.weight)),
                                      L.ptr(_f(ln.bias)), eps, int(relu), L.ptr(out), out_enc, L.ptr(out2), out2_enc or 0, st), 'srf_layernorm')
        return (out, out2) if out2_enc is not None else out
    fuse_ln = ln is not None and (n <= 128 or ln_per_tile)
    if ln is not None and not fuse_ln:
        tmp = alloc(L.F32)
        a.bias, a.out, a.out_enc = L.ptr(bias), L.ptr(tmp), L.F32
        L.check(lib.srf_linear(ctypes.byref(a), st), 'srf_linear')
        out = alloc(out_enc)
        out2 = alloc(out2_enc) if out2_enc is not None else None
        L.check(lib.srf_layernorm_enc(L.ptr(tmp), L.F32, m, n, 1, None, L.ptr(residual), L.ptr(_f(ln.weight)), L.ptr(_f(ln.bias)), eps,
                                      int(relu), L.ptr(out), out_enc, L.ptr(out2), out2_enc or 0, st), 'srf_layernorm')
        return (out, out2) if out2_enc is not None else out
    out = alloc(out_enc)
    out2 = alloc(out2_enc) if out2_enc is not None else None
    assert residual is None or out_enc == L.F32, 'a fused residual is read in the output encoding (fp32 here)'
    lnw = _f(ln.weight) if fuse_ln else None
    lnb = _f(ln.bias) if fuse_ln else None
    a.bias, a.residual = L.ptr(bias), L.ptr(residual)
    a.epi = (1 if relu else 0) | (2 if fuse_ln else 0)
    a.ln_w, a.ln_b, a.ln_per_tile = L.ptr(lnw), L.ptr(lnb), int(bool(ln_per_tile))
    a.out, a.out_enc, a.out2, a.out2_enc = L.ptr(out), out_enc, L.ptr(out2), out2_enc or 0
    L.check(lib.srf_linear(ctypes.byref(a), st), 'srf_linear')
    return (out, out2) if out2_enc is not None else out


class DynamicConv(nn.Module):
    def __init__(self, feat_channels, dynamic_dim=64, dynamic_num=2, pooler_resolution=7):
        super().__init__()
        assert dynamic_num == 2 and pooler_resolution == 7
        self.feat_channels = feat_channels
        self.dynamic_dim = dynamic_dim
        self.dynamic_num = dynamic_num
        self.num_params = feat_channels * dynamic_dim
        self.dynamic_layer = nn.Linear(feat_channels, dynamic_num * self.num_params)
        self.norm1 = nn.LayerNorm(dynamic_dim)
        self.norm2 = nn.LayerNorm(feat_channels)
        self.activation = nn.ReLU(inplace=True)
        self.out_layer = nn.Linear(feat_channels * pooler_resolution ** 2, feat_channels)
        self.norm3 = nn.LayerNorm(feat_channels)
        self._cache = {}

    def make_params(self, prop_feats, precision=None, prop_enc=None):
        """dynamic_layer(prop_feats): (K,C) -> (K, 2*C*d).  Depends only on the proposal features,
        so callers may run it concurrently with the RoI sampling of the same stage.  The split
        ('fp32') mode keeps the generated parameters in fp32 (the interaction kernel splits them)."""
        precision = precision or registry.get_precision()
        enc = registry.act_enc(precision)
        out_enc = L.F32 if (enc is None or L.enc_is_split(enc)) else enc
        x = prop_enc if (prop_enc is not None and enc is not None) else prop_feats
        return _linear(x, self.dynamic_layer, precision, self._cache, ('dyn', str(prop_feats.device)), out_enc=out_enc)

    def forward_kc(self, prop_feats, roi_feats, precision=None, params=None, prop_enc=None):
        """prop_feats (K,C) f32; roi_feats (K,49,C) f32 or (K,49,C|2C) in the mode's encoding
        (channel-last RoI features) -> (K,C) f32."""
        precision = precision or registry.get_precision()
        lib = L.load()
        k, c = prop_feats.shape
        d = self.dynamic_dim
        dev = prop_feats.device
        enc = registry.act_enc(precision)
        if params is None:
            params = self.make_params(prop_feats, precision, prop_enc=prop_enc)
        roi_feats = roi_feats.contiguous()
        if enc is not None and (c, d) not in ((128, 32), (256, 64)):
            # dims without a tensor-core interaction kernel: FFMA kernel on fp32 buffers
            roi_feats, params, enc = L.decode(roi_feats, c).contiguous(), L.decode(params, 2 * c * d).contiguous(), None
        out_enc = L.F32 if enc is None else enc
        inter = torch.empty((k, L.enc_width(out_enc, 49 * c)), dtype=L.enc_torch_dtype(out_enc), device=dev)
        L.check(lib.srf_dynconv_interact_tc(L.ptr(roi_feats), L.enc_of_tensor(roi_feats, c), L.ptr(params),
                                            L.enc_of_tensor(params, 2 * c * d), k, c, d, L.ptr(_f(self.norm1.weight)),
                                            L.ptr(_f(self.norm1.bias)), self.norm1.eps, L.ptr(_f(self.norm2.weight)),
                                            L.ptr(_f(self.norm2.bias)), self.norm2.eps, L.ptr(inter), out_enc, L.stream_ptr()),
                'srf_dynconv_interact')
        out = _linear(inter, self.out_layer, precision, self._cache, ('out', str(dev)), relu=True, ln=self.norm3, out_enc=L.F32)
        return out.float()

    def forward(self, prop_feats, roi_feats):
        """Reference signature: prop_feats (1, K, C), roi_feats (49, K, C) -> (K, C)."""
        return self.forward_kc(prop_feats[0], roi_feats.permute(1, 0, 2).contiguous())


class _SingleHeadBase(nn.Module):
    def _build_common(self, num_classes, feat_channels, pooler_resolution, use_focal_loss, use_fed_loss,
                      dim_feedforward, num_cls_convs, num_reg_convs, num_heads, dropout, scale_clamp, bbox_weights,
                      dynamic_conv, pc_range, voxel_size):
        self.feat_channels_lidar = feat_channels
        self.pc_range_lidar = pc_range
        self.voxel_size_lidar = voxel_size
        self.self_attn_lidar = nn.MultiheadAttention(feat_channels, num_heads, dropout=dropout)
        self.inst_interact_lidar = DynamicConv(feat_channels=feat_channels, pooler_resolution=pooler_resolution,
                                               dynamic_dim=dynamic_conv['dynamic_dim'],
                                               dynamic_num=dynamic_conv['dynamic_num'])
        self.linear1_lidar = nn.Linear(feat_channels, dim_feedforward)
        self.dropout_lidar = nn.Dropout(dropout)
        self.linear2_lidar = nn.Linear(dim_feedforward, feat_channels)
        self.norm1_lidar = nn.LayerNorm(feat_channels)
        self.norm2_lidar = nn.LayerNorm(feat_channels)
        self.norm3_lidar = nn.LayerNorm(feat_channels)
        self.dropout1_lidar = nn.Dropout(dropout)
        self.dropout2_lidar = nn.Dropout(dropout)
        self.dropout3_lidar = nn.Dropout(dropout)
        self.activation_lidar = nn.ReLU(inplace=True)

        def tower(n):
            mods = []
            for _ in range(n):
                mods += [nn.Linear(feat_channels, feat_channels, False), nn.LayerNorm(feat_channels), nn.ReLU(inplace=True)]
            return nn.ModuleList(mods)
        self.cls_module_lidar = tower(num_cls_convs)
        self.reg_module_lidar = tower(num_reg_convs)
        self.use_focal_loss = use_focal_loss
        self.use_fed_loss = use_fed_loss
        self.class_logits_lidar = nn.Linear(feat_channels, num_classes if (use_focal_loss or use_fed_loss) else num_classes + 1)
        self.bboxes_delta_lidar = nn.Linear(feat_channels, len(bbox_weights))
        self.scale_clamp = scale_clamp
        self.bbox_weights = bbox_weights

    # dense tail of a stage (SURVEY.md 8f rank 2): attention, interaction, FFN, towers, box update -- all on this
    # library's kernels (tcgen05 GEMMs with bias / residual / LayerNorm / ReLU epilogues, fp32 attention core)
    def _merged_towers(self, dev):
        """cls | reg towers as merged GEMMs (both are stacks of Linear(C, C, bias=False) + LayerNorm + ReLU, C = 128):
        layer 0 shares its input -> one (C -> 2C) GEMM; deeper layers pair up as block-diagonal (2C -> 2C) GEMMs; one
        LayerNorm per 128-column tile.  Returns [(view, ln_view, n_pairs)] or None when the shapes do not allow it."""
        C = self.feat_channels_lidar
        ncls, nreg = len(self.cls_module_lidar) // 3, len(self.reg_module_lidar) // 3
        if C != 128 or ncls < 1 or nreg < ncls:
            return None
        cache = self.__dict__.setdefault('_tail_cache', {})
        src = [p for mods in (self.cls_module_lidar, self.reg_module_lidar) for p in mods.parameters()]

        def make():
            layers = []
            for t in range(ncls):
                cl, rl = self.cls_module_lidar[3 * t], self.reg_module_lidar[3 * t]
                cn, rn = self.cls_module_lidar[3 * t + 1], self.reg_module_lidar[3 * t + 1]
                if t == 0:
                    w = torch.cat([cl.weight, rl.weight], 0)                      # (2C, C)
                else:
                    w = torch.zeros(2 * C, 2 * C, device=dev)
                    w[:C, :C], w[C:, C:] = cl.weight, rl.weight                     # block diagonal
                ln = nn.LayerNorm(C, eps=cn.eps)                                   # holder of the concatenated parameters
                ln.weight = nn.Parameter(torch.cat([cn.weight, rn.weight]).detach().to(dev), requires_grad=False)
                ln.bias = nn.Parameter(torch.cat([cn.bias, rn.bias]).detach().to(dev), requires_grad=False)
                assert cn.eps == rn.eps
                layers.append((_LinearView(w.detach().to(dev).contiguous(), None), ln))
            return layers
        return _cached(cache, ('towers', str(dev)), src, make)

    # dense tail of a stage (SURVEY.md 8f rank 2): attention, interaction, FFN, towers, box update -- all on this
    # library's kernels (tcgen05 GEMMs with bias / residual / LayerNorm / ReLU epilogues, fp32 attention core).
    # The fp32 trunk and the 16-bit operand of the next GEMM come out of the same epilogue (dual outputs).
    def _stage_tail(self, roi_feats_kc, bboxes, prop_feats, bs, n_p, precision=None):
        precision = precision or registry.get_precision()
        lib = L.load()
        C = self.feat_channels_lidar
        enc = registry.act_enc(precision)
        act = L.F32 if enc is None else enc
        cache = self.__dict__.setdefault('_tail_cache', {})
        dev = bboxes.device
        st = L.stream_ptr()
        k = bs * n_p
        x = _f(prop_feats.reshape(k, C))
        # self-attention over the proposals of a sample (srfdet_head.py:2281-2287)
        mha = self.self_attn_lidar
        qkv = _linear(x, _LinearView(mha.in_proj_weight, mha.in_proj_bias), precision, cache, 'in_proj', out_enc=L.F32)
        att = torch.empty((k, L.enc_width(act, C)), dtype=L.enc_torch_dtype(act), device=dev)
        L.check(lib.srf_mha_attention(L.ptr(qkv), bs, n_p, mha.num_heads, C // mha.num_heads, L.ptr(att), act, st), 'srf_mha_attention')
        prop, prop_e = _linear(att, mha.out_proj, precision, cache, 'out_proj', ln=self.norm1_lidar, residual=x, out_enc=L.F32, out2_enc=act)
        # instance interaction (:2289-2297)
        prop2 = self.inst_interact_lidar.forward_kc(prop, roi_feats_kc, precision, prop_enc=prop_e)
        obj = torch.empty_like(prop)
        obj_e = torch.empty((k, L.enc_width(act, C)), dtype=L.enc_torch_dtype(act), device=dev) if act != L.F32 else None
        L.check(lib.srf_layernorm_enc(L.ptr(prop2), L.F32, k, C, 1, None, L.ptr(prop), L.ptr(_f(self.norm2_lidar.weight)),
                                      L.ptr(_f(self.norm2_lidar.bias)), self.norm2_lidar.eps, 0, L.ptr(obj), L.F32, L.ptr(obj_e), act, st),
                'srf_layernorm')
        # FFN (:2299-2304)
        hid = _linear(obj_e if obj_e is not None else obj, self.linear1_lidar, precision, cache, 'ffn1', relu=True)
        obj, obj_e = _linear(hid, self.linear2_lidar, precision, cache, 'ffn2', ln=self.norm3_lidar, residual=obj, out_enc=L.F32, out2_enc=act)
        # towers (:2306-2313): (Linear(no bias), LayerNorm, ReLU) x n, then the two small projections
        merged = self._merged_towers(dev) if enc is not None else None
        if merged is not None:
            ncls = len(merged)
            f_e, f32 = obj_e, None
            for t, (lin, ln) in enumerate(merged):
                last = t == ncls - 1
                r = _linear(f_e, lin, precision, cache, ('tw', t), relu=True, ln=ln, ln_per_tile=True, out_enc=L.F32 if last else None,
                            out2_enc=act if last else None)
                f32, f_e = r if last else (None, r)
            cls_f = f32[:, :C].contiguous()
            reg_f, mods = None, self.reg_module_lidar
            nreg = len(mods) // 3
            if nreg == ncls:
                reg_f = f32[:, C:].contiguous()
            for t in range(ncls, nreg):                      # the regression tower is deeper: its remaining layers run alone
                lastr = t == nreg - 1
                a_cols = (C, 2 * C) if t == ncls else None
                reg_in = f_e if t == ncls else reg_in_next
                r = _linear(reg_in, mods[3 * t], precision, cache, ('reg', t), relu=True, ln=mods[3 * t + 1], out_enc=L.F32 if lastr else None,
                            a_cols=a_cols)
                if lastr:
                    reg_f = r
                else:
                    reg_in_next = r
        else:
            obj_in = obj_e if obj_e is not None else obj

            def tower(mods, tag):
                f = obj_in
                for t in range(0, len(mods), 3):
                    last = t + 3 >= len(mods)
                    f = _linear(f, mods[t], precision, cache, (tag, t), relu=True, ln=mods[t + 1], out_enc=L.F32 if last else None)
                return f if f.dtype == torch.float32 else L.decode(f, C)
            cls_f, reg_f = tower(self.cls_module_lidar, 'cls'), tower(self.reg_module_lidar, 'reg')
        logits = _linear(cls_f, self.class_logits_lidar, 'fp32_simt', cache, 'logits')
        deltas = _linear(reg_f, self.bboxes_delta_lidar, 'fp32_simt', cache, 'deltas')
        pred = self.apply_deltas_lidar(deltas, bboxes.view(-1, len(self.bbox_weights)))
        return logits.view(bs, n_p, -1), pred.view(bs, n_p, -1), obj

    def _stage_tail_torch(self, roi_feats_kc, bboxes, prop_feats, bs, n_p, precision=None):
        """The same rows as plain torch ops (cross-check of the kernel path in the tests)."""
        C = self.feat_channels_lidar
        prop = prop_feats.view(bs, n_p, C).permute(1, 0, 2)
        prop2 = self.self_attn_lidar(prop, prop, value=prop)[0]
        prop = self.norm1_lidar(prop + self.dropout1_lidar(prop2))
        prop = prop.permute(1, 0, 2).reshape(bs * n_p, C)
        prop2 = self.inst_interact_lidar.forward_kc(prop.contiguous(), roi_feats_kc, precision)
        obj = self.norm2_lidar(prop + self.dropout2_lidar(prop2))
        obj2 = self.linear2_lidar(self.dropout_lidar(self.activation_lidar(self.linear1_lidar(obj))))
        obj = self.norm3_lidar(obj + self.dropout3_lidar(obj2))
        cls_f, reg_f = obj.clone(), obj.clone()
        for layer in self.cls_module_lidar:
            cls_f = layer(cls_f)
        for layer in self.reg_module_lidar:
            reg_f = layer(reg_f)
        logits = self.class_logits_lidar(cls_f)
        deltas = self.bboxes_delta_lidar(reg_f)
        pred = self.apply_deltas_lidar(deltas, bboxes.view(-1, len(self.bbox_weights)))
        return logits.view(bs, n_p, -1), pred.view(bs, n_p, -1), obj

    def apply_deltas_lidar(self, deltas, boxes):
        """srfdet_head.py:2331-2420 (boxes carry ABSOLUTE centres after the in-place de-normalisation)."""
        deltas, boxes = _f(deltas), _f(boxes)
        k, dim = deltas.shape
        key = ('bbox_weights', str(deltas.device))
        cache = self.__dict__.setdefault('_tail_cache', {})
        if key not in cache:
            cache[key] = torch.tensor([float(v) for v in self.bbox_weights], dtype=torch.float32, device=deltas.device)
        out = torch.empty_like(deltas)
        L.check(L.load().srf_apply_deltas(L.ptr(deltas), L.ptr(boxes), k, dim, L.ptr(cache[key]), float(self.scale_clamp),
                                          L.f6(self.pc_range_lidar), L.ptr(out), L.stream_ptr()), 'srf_apply_deltas')
        return out


@HEADS.register_module()
class SingleSRFDetHeadLiDAR(_SingleHeadBase):
    def __init__(self, num_classes=80, feat_channels=256, pooler_resolution=7, use_focal_loss=True, use_fed_loss=False,
                 dim_feedforward=2048, num_cls_convs=1, num_reg_convs=3, num_heads=8, dropout=0.0,
                 scale_clamp=_DEFAULT_SCALE_CLAMP, bbox_weights=[1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 0.2, 0.2],
                 act_cfg=dict(type='ReLU', inplace=True), dynamic_conv=dict(dynamic_dim=64, dynamic_num=2),
                 pc_range=None, voxel_size=None, init_cfg=None, is_kitti=None):
        super().__init__()
        self._build_common(num_classes, feat_channels, pooler_resolution, use_focal_loss, use_fed_loss, dim_feedforward,
                           num_cls_convs, num_reg_convs, num_heads, dropout, scale_clamp, bbox_weights, dynamic_conv,
                           pc_range, voxel_size)

    def region_features(self, point_feats, bboxes, pooler):
        """RoI features, channel-last (bs*n_p, 49, C).  Mutates bboxes[..., :3] (reference :1638-1646)."""
        return points_feats_sampling_bboxes_roi(point_feats, bboxes, pooler, self.pc_range_lidar, self.voxel_size_lidar,
                                                channel_last=True)

    def forward(self, point_feats, bboxes, prop_feats, pooler, img_metas=None, precision=None):
        bs, n_p = bboxes.shape[:2]
        roi = self.region_features(point_feats, bboxes, pooler)
        if prop_feats is None:
            prop_feats = roi.mean(1).view(bs, n_p, -1)
        return self._stage_tail(roi, bboxes, prop_feats, bs, n_p, precision)


@HEADS.register_module()
class SingleSRFDetHead(_SingleHeadBase):
    def __init__(self, num_classes=80, feat_channels=256, pooler_resolution=7, use_focal_loss=True, use_fed_loss=False,
                 dim_feedforward=2048, num_cls_convs=1, num_reg_convs=3, num_heads=8, dropout=0.0,
                 scale_clamp=_DEFAULT_SCALE_CLAMP, bbox_weights=[1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 0.2, 0.2],
                 act_cfg=dict(type='ReLU', inplace=True), dynamic_conv=dict(dynamic_dim=64, dynamic_num=2),
                 pc_range=None, use_fusion=False, voxel_size=None, is_kitti=False, init_cfg=None):
        super().__init__()
        self.feat_channels = feat_channels
        self.use_fusion = use_fusion
        self.is_kitti = is_kitti
        self._build_common(num_classes, feat_channels, pooler_resolution, use_focal_loss, use_fed_loss, dim_feedforward,
                           num_cls_convs, num_reg_convs, num_heads, dropout, scale_clamp, bbox_weights, dynamic_conv,
                           pc_range, voxel_size)
        if use_fusion:
            self.output_fused_proj = nn.Linear(2 * feat_channels, feat_channels)
        self._cache = {}

    def region_features(self, img_feats, point_feats, bboxes, pooler, pooler_img, lidar2img, precision=None):
        """Fused RoI features (bs*n_p, 49, C) channel-last: image RoIs (each sample's own camera sum), BEV RoIs,
        concat + Linear(2C->C) (srfdet_head.py:2236-2264).  lidar2img (bs, n_cam, 4, 4), or (n_cam, 4, 4) at bs = 1."""
        precision = precision or registry.get_precision()
        img_roi = pts_roi = None
        if (self.use_fusion and img_feats is not None and point_feats is not None
                and maps_channels_last(flat_image_maps(img_feats), pooler_img.num_inputs)
                and maps_channels_last(point_feats, pooler.num_inputs)):
            # both samplers write their half of cat(img, pts) (srfdet_head.py:2257) in the GEMM's dtype
            k, c = bboxes.shape[0] * bboxes.shape[1], point_feats[0].shape[1]
            enc = registry.act_enc(precision)
            enc = L.F32 if enc is None else enc
            cat = torch.empty((k, 49, L.enc_width(enc, 2 * c)), device=bboxes.device, dtype=L.enc_torch_dtype(enc))
            img_feats_sampling_bboxes_roi(img_feats, bboxes, pooler_img, lidar2img, self.pc_range_lidar,
                                          channel_last=True, out=cat, ch_offset=0, out_enc=enc)
            points_feats_sampling_bboxes_roi(point_feats, bboxes, pooler, self.pc_range_lidar, self.voxel_size_lidar,
                                             channel_last=True, out=cat, ch_offset=c, out_enc=enc)
            fused = _linear(cat.view(k * 49, -1), self.output_fused_proj, precision, self._cache, ('fuse', str(cat.device)))
            return fused.view(k, 49, -1)
        if img_feats is not None:
            img_roi = img_feats_sampling_bboxes_roi(img_feats, bboxes, pooler_img, lidar2img, self.pc_range_lidar,
                                                    channel_last=True)
        if point_feats is not None:
            pts_roi = points_feats_sampling_bboxes_roi(point_feats, bboxes, pooler, self.pc_range_lidar,
                                                       self.voxel_size_lidar, channel_last=True)
        if img_roi is not None and pts_roi is not None and self.use_fusion:
            k = pts_roi.shape[0]
            cat = torch.cat((img_roi, pts_roi), dim=2).view(k * 49, -1)
            fused = _linear(cat, self.output_fused_proj, precision, self._cache, ('fuse', str(cat.device)))
            return fused.view(k, 49, -1)
        if not self.use_fusion and img_roi is not None and pts_roi is None:
            return img_roi
        if not self.use_fusion and pts_roi is not None and img_roi is None:
            return pts_roi
        raise ValueError('inconsistent fusion inputs')

    def forward(self, img_feats, point_feats, bboxes, prop_feats, pooler, img_metas, pooler_img=None, precision=None, lidar2img=None):
        bs, n_p = bboxes.shape[:2]
        if img_feats is not None and lidar2img is None:
            import numpy as np
            lidar2img = torch.as_tensor(np.asarray([m['lidar2img'] for m in img_metas]), dtype=torch.float32,
                                        device=bboxes.device)
        roi = self.region_features(img_feats, point_feats, bboxes, pooler, pooler_img, lidar2img, precision)
        if prop_feats is None:
            prop_feats = L.decode(roi, self.feat_channels).mean(1).view(bs, n_p, -1)
        return self._stage_tail(roi, bboxes, prop_feats, bs, n_p, precision)
