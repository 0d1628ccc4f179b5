"""ctypes binding of libsrfdet_b200.so (include/srfdet_b200.h).

There is NO CPU fallback: if the shared object is missing or a call fails, the op raises.
torch is used only to own device memory and streams; every kernel argument crosses the
boundary as a raw pointer / integer.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# SRFDET_B200_LIB: development variants of the same library (e.g. the -DSRF_IGEMM_PROF build)
SO_PATH = os.environ.get('SRFDET_B200_LIB') or os.path.join(_HERE, 'csrc', 'libsrfdet_b200.so')

F32, BF16, F16, BF16X2, F16X2 = 0, 1, 2, 3, 4      # include/srfdet_b200.h element encodings


def enc_is_split(enc):
    return enc in (BF16X2, F16X2)


def enc_torch_dtype(enc):
    """torch dtype of the buffer that holds encoding `enc` (split rows are 2c elements wide)."""
    import torch
    return {F32: torch.float32, BF16: torch.bfloat16, F16: torch.float16, BF16X2: torch.bfloat16, F16X2: torch.float16}[enc]


def enc_width(enc, c):
    return 2 * c if enc_is_split(enc) else c


def enc_of_tensor(t, c):
    """Encoding of a tensor whose logical row has c values (last dim c or 2c)."""
    import torch
    if t.dtype == torch.float32:
        return F32
    split = t.shape[-1] == 2 * c
    return {torch.bfloat16: (BF16, BF16X2), torch.float16: (F16, F16X2)}[t.dtype][int(split)]


def decode(t, c):
    """fp32 view of an encoded tensor (tests / debugging)."""
    if t.shape[-1] == 2 * c and t.dtype != __import__('torch').float32:
        return t[..., :c].float() + t[..., c:].float()
    return t.float()


class SrfError(RuntimeError):
    pass


class Geom(Structure):
    _fields_ = [('vs', c_float * 3), ('lo', c_float * 3), ('hi', c_float * 3), ('grid', c_int32 * 3)]


class VfeParams(Structure):
    _fields_ = [('pos_w0', c_void_p), ('pos_b0', c_void_p), ('pos_w1', c_void_p), ('pos_b1', c_void_p),
                ('vfe_w0', c_void_p), ('vfe_b0', c_void_p), ('vfe_w1', c_void_p), ('vfe_b1', c_void_p),
                ('cin', c_int32), ('c0', c_int32), ('c1', c_int32),
                ('vx', c_float), ('vy', c_float), ('vz', c_float),
                ('x_off', c_float), ('y_off', c_float), ('z_off', c_float)]


class ConvArgs(Structure):
    _fields_ = [('in_', c_void_p), ('in_dtype', c_int32), ('in_rows', c_int32), ('cin', c_int32), ('cout', c_int32), ('kvol', c_int32),
                ('nbr', c_void_p), ('tile_mask', c_void_p), ('cap_out', c_int32), ('d_n_out', c_void_p),
                ('w', c_void_p), ('bias', c_void_p), ('residual', c_void_p), ('relu', c_int32),
                ('out', c_void_p), ('out_dtype', c_int32), ('dense', c_void_p), ('out_coors', c_void_p),
                ('out_dims', c_int32 * 4)]


class RoiOut(Structure):
    _fields_ = [('ptr', c_void_p), ('channel_last', c_int32), ('dtype', c_int32), ('row_stride', c_int32), ('ch_offset', c_int32)]


class Pyramid(Structure):
    _fields_ = [('feat', c_void_p * 4), ('h', c_int32 * 4), ('w', c_int32 * 4), ('stride', c_float * 4),
                ('n_levels', c_int32), ('channels', c_int32), ('channels_last', c_int32)]


class LinearArgs(Structure):
    _fields_ = [('a', c_void_p), ('a_enc', c_int32), ('m', c_int32), ('k', c_int32), ('a_stride', c_int64), ('a_lo_off', c_int64),
                ('w', c_void_p), ('n', c_int32), ('bias', c_void_p), ('residual', c_void_p), ('epi', c_int32), ('ln_w', c_void_p),
                ('ln_b', c_void_p), ('ln_eps', c_float), ('ln_per_tile', c_int32), ('out', c_void_p), ('out_enc', c_int32),
                ('out2', c_void_p), ('out2_enc', c_int32), ('k_splits', c_int32)]


class Rows(Structure):
    _fields_ = [('src', c_void_p), ('dst', c_void_p), ('src_ld', c_int32), ('dst_ld', c_int32), ('width', c_int32)]


class SweepSrc(Structure):
    _fields_ = [('points', c_void_p), ('cap', c_int32), ('ld', c_int32), ('flags', c_int32)]


SWEEP_TRANSFORM, SWEEP_TIME_LAG, SWEEP_REMOVE_CLOSE = 1, 2, 4      # include/srfdet_b200.h srf_sweep_src flags
SWEEP_MAX_SOURCES, SWEEP_MAX_COLS = 64, 8


class Map(Structure):
    _fields_ = [('ptr', c_void_p), ('c', c_int32), ('sn', c_int64), ('sc', c_int64), ('sh', c_int64), ('sw', c_int64)]


def map_view(t):
    """srf_map of a (n, c, h, w) fp32 CUDA tensor in whatever memory format it has (NCHW or channels_last)."""
    assert t.dim() == 4 and t.is_cuda and str(t.dtype) == 'torch.float32'
    sn, sc, sh, sw = t.stride()
    return Map(t.data_ptr(), t.shape[1], sn, sc, sh, sw)


_I4 = c_int32 * 4
_I3 = c_int32 * 3
_F3 = c_float * 3
_F6 = c_float * 6

# name -> (restype, argtypes).  Every symbol of include/srfdet_b200.h is listed here; the
# CPU test-suite checks the two stay in sync and that the library exports all of them.
PROTOTYPES = {
    'srf_version': (c_int32, []),
    'srf_last_error': (c_char_p, []),
    'srf_sm_count': (c_int32, []),
    'srf_conv3x3_last_used_tma': (c_int32, []),
    'srf_launch_count': (ctypes.c_uint64, []),
    'srf_geom_init': (c_int32, [POINTER(Geom), POINTER(c_float), POINTER(c_float)]),
    'srf_dynamic_voxelize': (c_int32, [c_void_p, c_int32, c_int32, POINTER(Geom), c_int32, c_void_p, c_void_p]),
    'srf_hard_voxelize_ws_bytes': (c_size_t, [c_int32, c_int32, c_int32]),
    'srf_hard_voxelize': (c_int32, [c_void_p, c_int32, c_int32, POINTER(Geom), c_int32, c_int32, c_int32, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'srf_concat_counted_rows': (c_int32, [c_void_p, c_int32, c_int32, POINTER(Rows), c_int32, c_void_p, c_void_p]),
    'srf_index_bytes': (c_size_t, [c_int64]),
    'srf_index_clear': (c_int32, [c_void_p, c_int64, c_void_p]),
    'srf_index_mark': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p, c_void_p]),
    'srf_index_mark_strided': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p, POINTER(c_int32),
                                         POINTER(c_int32), POINTER(c_int32), c_void_p]),
    'srf_index_finalize': (c_int32, [c_void_p, c_int64, c_void_p, c_void_p]),
    'srf_index_emit_coors': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p]),
    'srf_index_lookup': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    'srf_index_perm': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    'srf_gather_rows': (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_scatter_ws_bytes': (c_size_t, [c_int64, c_int32, c_int32]),
    'srf_dynamic_scatter': (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, POINTER(c_int32), c_int32,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'srf_dynamic_vfe_ws_bytes': (c_size_t, [c_int64, c_int32]),
    'srf_dynamic_vfe': (c_int32, [c_void_p, c_void_p, c_int32, POINTER(c_int32), POINTER(VfeParams), c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'srf_pillar_vfe': (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32,
                                 POINTER(c_float), POINTER(c_float), c_int32, c_void_p, c_void_p]),
    'srf_pillars_scatter': (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_pillar_encode_rows': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                         c_void_p, c_int32, POINTER(c_float), POINTER(c_float), c_int32, c_int32, c_int32,
                                         c_int32, c_void_p, c_void_p]),
    'srf_dense_rulebook': (c_int32, [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    'srf_nchw_to_rows': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_upsample_add': (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    'srf_rulebook_build': (c_int32, [c_void_p, POINTER(c_int32), c_void_p, c_void_p, c_int32, c_void_p,
                                     POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_void_p, c_void_p, c_void_p]),
    'srf_conv3x3_rows': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'srf_spconv_f32': (c_int32, [POINTER(ConvArgs), c_void_p]),
    'srf_spconv_bf16': (c_int32, [POINTER(ConvArgs), c_void_p]),
    'srf_spconv_tc': (c_int32, [POINTER(ConvArgs), c_void_p]),
    'srf_pack_weight_tc': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_convert_rows': (c_int32, [c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_pack_weight_bf16': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_f32_to_bf16': (c_int32, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_linear_tile_k': (c_int32, [c_int32]),
    'srf_linear_tile_n': (c_int32, [c_int32]),
    'srf_linear_tile_k_enc': (c_int32, [c_int32, c_int32]),
    'srf_linear_splits_enc': (c_int32, [c_int32, c_int32, c_int32]),
    'srf_pack_linear_tc': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_linear': (c_int32, [POINTER(LinearArgs), c_void_p]),
    'srf_linear_tc': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_void_p,
                                c_void_p, c_float, c_void_p, c_int32, c_int32, c_void_p]),
    'srf_layernorm_enc': (c_int32, [c_void_p, c_int32, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                                    c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'srf_mha_attention': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    'srf_apply_deltas': (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_float, POINTER(c_float), c_void_p, c_void_p]),
    'srf_dwconv3x3_s2': (c_int32, [POINTER(Map), POINTER(Map), c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_channel_sum': (c_int32, [POINTER(Map), POINTER(Map), c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_gemv_f32': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
    'srf_dpg_mix': (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p,
                              c_void_p, c_int32, c_void_p]),
    'srf_decode_boxes': (c_int32, [c_void_p, c_int64, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    'srf_dynconv_interact_tc': (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                          c_float, c_void_p, c_void_p, c_float, c_void_p, c_int32, c_void_p]),
    'srf_pack_linear_bf16': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_linear_bf16': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p,
                                  c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    'srf_linear_f32': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
    'srf_layernorm': (c_int32, [c_void_p, c_int32, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_float, c_int32, c_void_p, c_void_p]),
    'srf_linear_splits': (c_int32, [c_int32, c_int32]),
    'srf_boxes_to_corners': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_roi_extract': (c_int32, [POINTER(Pyramid), c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'srf_bev_roi_features': (c_int32, [POINTER(Pyramid), c_void_p, c_int32, c_int32, c_int32, POINTER(c_float),
                                       POINTER(c_float), c_int32, POINTER(RoiOut), c_void_p, c_void_p]),
    'srf_img_roi_features': (c_int32, [POINTER(Pyramid), c_void_p, c_int32, c_int32, c_void_p, c_int32,
                                       POINTER(c_float), POINTER(RoiOut), c_void_p, c_void_p]),
    'srf_dynconv_interact': (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    'srf_iou_bev': (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    'srf_nms_bev_ws_bytes': (c_size_t, [c_int32, c_int32, c_int32]),
    'srf_nms_bev': (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_float, c_float, c_int32, c_int32,
                              POINTER(c_float), c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'srf_merge_sweeps_ws_bytes': (c_size_t, [POINTER(SweepSrc), c_int32]),
    'srf_merge_sweeps': (c_int32, [POINTER(SweepSrc), c_int32, c_void_p, c_void_p, c_void_p, POINTER(c_int32), c_int32,
                                   POINTER(c_float), c_float, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
}

_lib = None


def load():
    """Load the shared object (raises SrfError when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise SrfError(f'{SO_PATH} not found: build it with `python -m srfdet_b200.build` '
                           '(there is no CPU fallback)')
        lib = ctypes.CDLL(SO_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = load().srf_last_error()
        raise SrfError(f'{what} failed (rc={rc}): {msg.decode() if msg else "?"}')


def ptr(t):
    """Raw device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), 'kernel arguments must be contiguous CUDA tensors'
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def i4(v):
    return _I4(*[int(x) for x in v])


def i3(v):
    return _I3(*[int(x) for x in v])


def f3(v):
    return _F3(*[float(x) for x in v])


def f6(v):
    return _F6(*[float(x) for x in v])


def make_geom(voxel_size, pc_range):
    """Host-side srf_geom (same fp32 arithmetic as srf_geom_init: grid = rint((hi - lo) / vs), half
    to even).  Pure Python on purpose: constructing the drop-in modules must not load the CUDA
    library (bench.py's reference arm builds the same seeded weights on a host without using it)."""
    import numpy as np
    g = Geom()
    for j in range(3):
        vs, lo, hi = np.float32(voxel_size[j]), np.float32(pc_range[j]), np.float32(pc_range[3 + j])
        g.vs[j], g.lo[j], g.hi[j] = float(vs), float(lo), float(hi)
        g.grid[j] = int(np.rint(np.float32(np.float32(hi - lo) / vs)))
        if g.grid[j] <= 0:
            raise SrfError(f'empty grid on axis {j}')
    return g


def make_geom_c(voxel_size, pc_range):
    """The same through the library's srf_geom_init (parity of the two is tested)."""
    g = Geom()
    check(load().srf_geom_init(ctypes.byref(g), f3(voxel_size), f6(pc_range)), 'srf_geom_init')
    return g
