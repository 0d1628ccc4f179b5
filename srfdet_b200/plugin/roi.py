"""Region-feature sampling: bbox2roi / SingleRoIExtractor (mmdet 2.28.2 names, built from
cfg `roi_extractor_lidar` / `roi_extractor_img`, configs/nus/srfdet_voxel_nusc_LC.py:169-178),
boxes3d_to_corners3d (mmdet3d_plugin/core/bbox/util.py:84-176) and the fused samplers
that replace points_feats_sampling_bboxes_roi / img_feats_sampling_bboxes_roi
(mmdet3d_plugin/models/sparse_heads/srfdet_head.py:2568-2629, 2424-2565)."""
import ctypes

import torch
from torch import nn

from .. import _lib as L
from .registry import ROI_EXTRACTORS


def bbox2roi(bbox_list):
    """mmdet.core.bbox2roi: list of (n,4+) boxes per image -> (sum n, 5) [img_idx, x1,y1,x2,y2]."""
    out = []
    for i, b in enumerate(bbox_list):
        out.append(torch.cat([b.new_full((b.size(0), 1), i), b[:, :4]], dim=-1))
    return torch.cat(out, 0)


def maps_channels_last(feats, n_levels=None):
    """True when every level is a torch.channels_last tensor (NHWC in memory) the coalesced
    kernels consume in place."""
    n_levels = len(feats) if n_levels is None else min(n_levels, len(feats))
    c = feats[0].shape[-3]
    return c % 4 == 0 and c <= 256 and all(
        f.dim() == 4 and f.shape[1] > 1 and not f.is_contiguous() and f.is_contiguous(memory_format=torch.channels_last)
        for f in feats[:n_levels])


def _pyramid(feats, strides, n_levels):
    p = L.Pyramid()
    n_levels = min(n_levels, len(feats))
    c = feats[0].shape[-3]
    keep = []
    cl = maps_channels_last(feats, n_levels)
    p.channels_last = int(cl)
    for l in range(n_levels):
        f = feats[l]
        assert f.dtype == torch.float32 and f.shape[-3] == c, 'feature maps must be fp32 with equal channels'
        if not cl:
            f = f.contiguous()
        keep.append(f)
        p.feat[l] = f.data_ptr()
        p.h[l], p.w[l] = f.shape[-2], f.shape[-1]
        p.stride[l] = float(strides[l])
    p.n_levels = n_levels
    p.channels = c
    return p, keep


def boxes3d_to_corners3d(boxes3d, bottom_center=False, ry=False):
    """(bs, N, >=8) [cx,cy,cz,log w,log l,log h,sin,cos] -> (bs, N, 8, 3)."""
    if bottom_center or ry:
        raise NotImplementedError('only the (bottom_center=False, ry=False) form used by the head is built')
    b = boxes3d.contiguous().float()
    bs, n, d = b.shape
    out = torch.empty((bs, n, 8, 3), dtype=torch.float32, device=b.device)
    L.check(L.load().srf_boxes_to_corners(L.ptr(b), bs * n, d, L.ptr(out), L.stream_ptr()), 'srf_boxes_to_corners')
    return out


@ROI_EXTRACTORS.register_module()
class SingleRoIExtractor(nn.Module):
    """mmdet SingleRoIExtractor over mmcv RoIAlign (avg, aligned=True); finest_scale 56.

    forward(feats: list[(N,C,H,W) f32], rois (K,5)) -> (K, C, 7, 7)."""

    def __init__(self, roi_layer, out_channels, featmap_strides, finest_scale=56, init_cfg=None):
        super().__init__()
        cfg = dict(roi_layer)
        t = cfg.pop('type')
        assert t == 'RoIAlign', 'only RoIAlign is built'
        self.output_size = cfg.get('output_size', 7)
        self.sampling_ratio = cfg.get('sampling_ratio', 0)
        if self.output_size != 7 or self.sampling_ratio != 2 or finest_scale != 56 \
                or cfg.get('pool_mode', 'avg') != 'avg' or not cfg.get('aligned', True):
            raise NotImplementedError('kernels are specialised to RoIAlign(7, sampling_ratio=2, avg, aligned), '
                                      'finest_scale=56 (the reference configs)')
        self.out_channels = out_channels
        self.featmap_strides = list(featmap_strides)
        self.finest_scale = finest_scale

    @property
    def num_inputs(self):
        return len(self.featmap_strides)

    def forward(self, feats, rois, roi_scale_factor=None, channel_last=False):
        assert roi_scale_factor is None
        rois = rois.contiguous().float()
        k = rois.shape[0]
        p, keep = _pyramid(feats, self.featmap_strides, self.num_inputs)
        c = p.channels
        out = torch.empty((k, 49, c) if channel_last else (k, c, 7, 7), dtype=torch.float32, device=rois.device)
        L.check(L.load().srf_roi_extract(ctypes.byref(p), L.ptr(rois), k, L.ptr(out), int(channel_last), L.stream_ptr()),
                'srf_roi_extract')
        return out


def _roi_out(k, c, channel_last, device, out=None, ch_offset=0, out_enc=None):
    """Destination spec: a fresh (k,C,7,7) / (k,49,C) fp32 tensor, or a caller-provided
    channel-last (k,49,C') buffer in encoding `out_enc` (fp32, bf16, f16, or a split form whose rows
    are [hi(C'/2) | lo(C'/2)]) filled at channel offset `ch_offset`."""
    if out is None:
        out = torch.empty((k, 49, c) if channel_last else (k, c, 7, 7), dtype=torch.float32, device=device)
        spec = L.RoiOut(out.data_ptr(), int(channel_last), L.F32, c, 0)
    else:
        assert out.is_contiguous() and out.dim() == 3 and out.shape[0] == k and out.shape[1] == 49
        if out_enc is None:
            out_enc = {torch.float32: L.F32, torch.bfloat16: L.BF16, torch.float16: L.F16}[out.dtype]
        assert out.dtype == L.enc_torch_dtype(out_enc)
        spec = L.RoiOut(out.data_ptr(), 1, out_enc, out.shape[2], int(ch_offset))
    return out, spec


def points_feats_sampling_bboxes_roi(points_feats, bboxes, pooler, pc_range, voxel_size, channel_last=False,
                                     return_rois=False, out=None, ch_offset=0, mutate=True, out_enc=None):
    """Fused srfdet_head.py:2568-2629.  bboxes (bs, n_p, >=8) normalised centres; the
    centres are de-normalised IN PLACE like the reference (:2587) unless mutate=False.
    -> (bs*n_p, C, 7, 7) (or channel-last (bs*n_p, 49, C); `out`/`ch_offset`: write into a slice
    of a caller buffer)."""
    assert bboxes.is_contiguous() and bboxes.dtype == torch.float32
    bs, n_p, d = bboxes.shape
    p, keep = _pyramid(points_feats, pooler.featmap_strides, pooler.num_inputs)
    c = p.channels
    k = bs * n_p
    out, spec = _roi_out(k, c, channel_last, bboxes.device, out, ch_offset, out_enc)
    rois = torch.empty((k, 5), dtype=torch.float32, device=bboxes.device) if return_rois else None
    L.check(L.load().srf_bev_roi_features(ctypes.byref(p), L.ptr(bboxes), bs, n_p, d, L.f6(pc_range), L.f3(voxel_size), int(bool(mutate)),
                                          ctypes.byref(spec), L.ptr(rois), L.stream_ptr()), 'srf_bev_roi_features')
    return (out, rois) if return_rois else out


def flat_image_maps(img_feats):
    """(B, n_cam, C, H, W) image maps per level -> (B*n_cam, C, H, W): image b*n_cam + cam is camera cam of sample b.
    A view where the strides allow one (the head's img_convs outputs and any densely packed level); a level whose images
    are not evenly spaced is copied."""
    for f in img_feats:
        if f.dim() != 5:
            raise ValueError(f'image maps must be (B, n_cam, C, H, W) per level, got {tuple(f.shape)}')
    return [f.reshape(-1, *f.shape[2:]) for f in img_feats]


def img_feats_sampling_bboxes_roi(img_feats, bboxes, pooler, lidar2img, pc_range, channel_last=False,
                                  return_rois=False, out=None, ch_offset=0, out_enc=None):
    """Fused srfdet_head.py:2424-2565 over B samples, each with the reference's batch-1 semantics (SURVEY.md 3.4: a
    batch of B fusion samples is B independent batch-1 calls): sample b sums its own cameras, projected by its own
    lidar2img[b].  img_feats: list of (B, n_cam, C, H, W); bboxes (B, n_p, >=8) (not mutated); lidar2img
    (B, n_cam, 4, 4) tensor, or (n_cam, 4, 4) at B = 1.  -> (B*n_p, C, 7, 7) (or channel-last (B*n_p, 49, C); `out` /
    `ch_offset`: write into a slice of a caller buffer); return_rois: also the (B*n_cam*n_p, 5) image RoIs, row
    (b*n_cam + cam)*n_p + p with column 0 = b*n_cam + cam (srf_roi_extract on the flattened maps reads them)."""
    bs, n_p, d = bboxes.shape
    flat = flat_image_maps(img_feats)
    if any(f.shape[0] != bs for f in img_feats):
        raise ValueError(f'image maps of batch {[f.shape[0] for f in img_feats]} for {bs} samples of boxes')
    n_cam = img_feats[0].shape[1]
    if any(f.shape[1] != n_cam for f in img_feats):
        raise ValueError('every image level needs the same number of cameras')
    if tuple(lidar2img.shape) not in ((bs, n_cam, 4, 4),) + (((n_cam, 4, 4),) if bs == 1 else ()):
        raise ValueError(f'lidar2img {tuple(lidar2img.shape)} does not match {bs} sample(s) of {n_cam} cameras: '
                         f'pass ({bs}, {n_cam}, 4, 4)')
    b = bboxes.contiguous().float()
    p, keep = _pyramid(flat, pooler.featmap_strides, pooler.num_inputs)
    l2i = lidar2img.reshape(bs, n_cam, 4, 4).contiguous().float()
    c = p.channels
    out, spec = _roi_out(bs * n_p, c, channel_last, b.device, out, ch_offset, out_enc)
    rois = torch.empty((bs * n_cam * n_p, 5), dtype=torch.float32, device=b.device) if return_rois else None
    L.check(L.load().srf_img_roi_features(ctypes.byref(p), L.ptr(b), bs, n_p, d, L.ptr(l2i), n_cam, L.f6(pc_range),
                                          ctypes.byref(spec), L.ptr(rois), L.stream_ptr()), 'srf_img_roi_features')
    return (out, rois) if return_rois else out
