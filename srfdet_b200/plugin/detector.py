"""The SRFDet detector (mmdet3d_plugin/models/detectors/srfdet.py) built from the reference's unmodified
`model` config dict.

`SRFDetPointPath`: the point-cloud side, `voxelize` (:204-247) and `extract_point_features` (:249-276) up to the
middle encoder.  Pillar configs (PillarFeatureNetCustom + PointPillarsScatter) are recognised from the modules the config
builds; `pillar_rows` takes them straight to the backbone's input rows (srf_pillar_encode_rows), with no canvas.  `SRFDet` / `SRFDetWaymo` (registry names of the reference, srfdet.py / srfdetwaymo.py): the whole
detector above it -- point path, SECONDCustom + FPN (`pts_backbone`, `pts_neck`) and SRFDetHead (`bbox_head`) --
with the reference's test-time call contract (`forward_test` / `simple_test`), checkpoint loading by the reference's
attribute names and a device-resident, optionally graph-captured `infer`.  The image backbone and image neck are not
built: callers pass the image-neck outputs (DESIGN.md §1).  Camera-fusion configs take batches too: a batch of B fusion
samples is B independent batch-1 calls of the reference (SURVEY.md §3.4), each sample with its own image maps and its own
lidar2img.
"""
import collections
import os

import numpy as np
import torch
from torch import nn

from .. import _lib as L
from . import registry
from .ops import Voxelization
from .pillar import PillarFeatureNetCustom, PointPillarsScatter
from .registry import DETECTORS, build_backbone, build_head, build_middle_encoder, build_neck, build_voxel_encoder
from .voxel_encoder import HardSimpleVFE


class SRFDetPointPath(nn.Module):
    def __init__(self, pts_voxel_layer=None, pts_voxel_encoder=None, pts_middle_encoder=None, **unused):
        super().__init__()
        self.pts_voxel_layer_cfg = dict(pts_voxel_layer)
        self.pts_voxel_layer = Voxelization(**pts_voxel_layer)
        self.pts_voxel_encoder = build_voxel_encoder(pts_voxel_encoder)
        self.pts_middle_encoder = build_middle_encoder(pts_middle_encoder)
        self.unused_cfg = unused
        self.eval()

    @classmethod
    def from_config(cls, path_or_model):
        model = registry.load_config(path_or_model)['model'] if isinstance(path_or_model, str) else dict(path_or_model)
        model = dict(model)
        model.pop('type', None)
        enc = dict(model['pts_middle_encoder'])
        enc.pop('init_cfg', None)   # checkpoints are loaded explicitly (no network / ckpts here)
        model['pts_middle_encoder'] = enc
        return cls(**model)

    @property
    def is_dynamic(self):
        return self.pts_voxel_layer_cfg['max_num_points'] == -1

    @property
    def is_pillar(self):
        return isinstance(self.pts_voxel_encoder, PillarFeatureNetCustom) and isinstance(self.pts_middle_encoder, PointPillarsScatter)

    @torch.no_grad()
    def hard_voxel_blocks(self, points, want_voxels=False, want_mean=False):
        """Hard voxelization of B clouds without a host read: sample i fills block i of max_voxels rows.
        -> dict(voxels (B, M, T, C) | None, num_points (B, M), coors (B, M, 4) bzyx, mean (B, M, C) | None,
        count (B,) int32 device); rows past a block's count are unspecified."""
        assert not self.is_dynamic
        bs, c, dev = len(points), points[0].shape[1], points[0].device
        if any(p.shape[1] != c for p in points):
            raise ValueError('all clouds of a batch need the same number of point features')
        mv = int(self.pts_voxel_layer._max_voxels())
        if mv <= 0:
            mv = max(max(p.shape[0] for p in points), 1)
        T = int(self.pts_voxel_layer.max_num_points)
        blk = dict(voxels=torch.empty((bs, mv, T, c), dtype=torch.float32, device=dev) if want_voxels else None,
                   num_points=torch.empty((bs, mv), dtype=torch.int32, device=dev),
                   coors=torch.empty((bs, mv, 4), dtype=torch.int32, device=dev),
                   mean=torch.empty((bs, mv, c), dtype=torch.float32, device=dev) if want_mean else None,
                   count=torch.zeros((bs,), dtype=torch.int32, device=dev))
        for i, p in enumerate(points):
            self.pts_voxel_layer.hard_padded(p, batch_idx=i, want_voxels=want_voxels, want_mean=want_mean,
                                             out={k: None if v is None else v[i:i + 1] if k == 'count' else v[i]
                                                  for k, v in blk.items()})
        return blk

    @torch.no_grad()
    def pillar_rows(self, points, enc):
        """Pillar configs: B clouds -> the first backbone convolution's input pixel rows in encoding enc, through
        PillarFeatureNetCustom.encode_rows (PFN + PointPillarsScatter + row encoding in one kernel) without a host read.
        -> (rows (>= B*ny*nx, enc_width(enc, C)), ny, nx)."""
        blk = self.hard_voxel_blocks(points, want_voxels=True)
        ny, nx = self.pts_middle_encoder.ny, self.pts_middle_encoder.nx
        rows = self.pts_voxel_encoder.encode_rows(blk['voxels'], blk['num_points'], blk['coors'], blk['count'], ny, nx, enc)
        return rows, ny, nx

    @torch.no_grad()
    def voxelize(self, points):
        """Reference contract (host-synchronising, like srfdet.py:204-247).
        hard   : (voxels (M,T,C), num_points (M,), coors (M,4))
        dynamic: (points (sum N, C), coors (sum N, 4))"""
        if not self.is_dynamic:
            vs, cs, ns = [], [], []
            for i, res in enumerate(points):
                o = self.pts_voxel_layer.hard_padded(res, batch_idx=i)
                m = int(o['count'].item())
                vs.append(o['voxels'][:m])
                cs.append(o['coors'][:m])
                ns.append(o['num_points'][:m])
            return torch.cat(vs, 0), torch.cat(ns, 0), torch.cat(cs, 0)
        coors = [self.pts_voxel_layer.dynamic(res, batch_idx=i) for i, res in enumerate(points)]
        return torch.cat(points, 0), torch.cat(coors, 0)

    @torch.no_grad()
    def extract_point_features(self, points, precision=None):
        """points: list of (N_i, C) fp32 CUDA tensors -> dense BEV (B, C*D, H, W) fp32.
        Single-frame inputs (all reference test configs use batch 1) run without any host
        synchronisation: voxel counts stay on the device end to end."""
        bs = len(points)
        if not self.is_dynamic:
            if self.is_pillar:      # the modules' own kernels, one launch each per block with that block's device count
                blk = self.hard_voxel_blocks(points, want_voxels=True)
                mid = self.pts_middle_encoder
                canvas = torch.empty((bs, self.pts_voxel_encoder.pfn_layers[0].units, mid.ny, mid.nx), device=points[0].device,
                                     memory_format=torch.channels_last if mid.channels_last else torch.contiguous_format).zero_()
                for i in range(bs):
                    n = blk['count'][i:i + 1]
                    feats = self.pts_voxel_encoder(blk['voxels'][i], blk['num_points'][i], blk['coors'][i], num_voxels=n)
                    mid.scatter_into(canvas, feats, blk['coors'][i], num_voxels=n)
                return canvas
            if bs == 1 and isinstance(self.pts_voxel_encoder, HardSimpleVFE):
                o = self.pts_voxel_layer.hard_padded(points[0], batch_idx=0, want_voxels=False, want_mean=True)
                c = self.pts_voxel_encoder.num_features
                mean = o['mean'] if o['mean'].shape[1] == c else o['mean'][:, :c].contiguous()
                return self.pts_middle_encoder(mean, o['coors'], 1, num_voxels=o['count'], precision=precision)
            voxels, num_points, coors = self.voxelize(points)
            feats = self.pts_voxel_encoder(voxels, num_points, coors)
            return self.pts_middle_encoder(feats, coors, bs, precision=precision)
        pts, coors = self.voxelize(points)
        vf, vc, count = self.pts_voxel_encoder.forward_padded(pts, coors, batch_size=bs)
        return self.pts_middle_encoder(vf, vc, bs, num_voxels=count, precision=precision)


def _drop_init_cfg(cfg):
    """Config with every init_cfg / pretrained entry removed at any depth: weights come from load_checkpoint only."""
    if isinstance(cfg, dict):
        return {k: _drop_init_cfg(v) for k, v in cfg.items() if k not in ('init_cfg', 'pretrained')}
    if isinstance(cfg, (list, tuple)):
        return type(cfg)(_drop_init_cfg(v) for v in cfg)
    return cfg


CheckpointKeys = collections.namedtuple('CheckpointKeys', ['missing_keys', 'unexpected_keys', 'set_aside_keys'])
_IMAGE_PREFIXES = ('img_backbone.', 'img_neck.')


@DETECTORS.register_module(name='SRFDet')
class SRFDet(SRFDetPointPath):
    """SRFDet (srfdet.py:18-77 constructor, :141-173 extract_feat, :249-340 forward_test / simple_test), inference only.

    Attributes keep the reference's names, so its checkpoints load unchanged: pts_voxel_layer, pts_voxel_encoder,
    pts_middle_encoder, pts_backbone, pts_neck, bbox_head.  img_backbone / img_neck configs are kept (not built) in
    `img_backbone_cfg` / `img_neck_cfg`.  use_graph=True: `infer` is captured into one CUDA graph per
    (batch size, point counts, precision, image-map shapes and strides, lidar2img shape) and replayed; outputs then live
    in graph-owned buffers that the next replay overwrites.  A graph bakes in the weights it was captured with: loading weights through this
    module (load_checkpoint / load_state_dict) drops the captured graphs, any other weight change needs reset_graphs()."""

    def __init__(self, pts_voxel_layer=None, pts_voxel_encoder=None, pts_middle_encoder=None, pts_backbone=None,
                 pts_neck=None, bbox_head=None, img_backbone=None, img_neck=None, train_cfg=None, test_cfg=None,
                 use_graph=False, **unused):
        cfg = _drop_init_cfg(dict(pts_voxel_layer=pts_voxel_layer, pts_voxel_encoder=pts_voxel_encoder,
                                  pts_middle_encoder=pts_middle_encoder, pts_backbone=pts_backbone, pts_neck=pts_neck,
                                  bbox_head=bbox_head, img_backbone=img_backbone, img_neck=img_neck, test_cfg=test_cfg))
        unused = _drop_init_cfg(unused)
        super().__init__(cfg['pts_voxel_layer'], cfg['pts_voxel_encoder'], cfg['pts_middle_encoder'], **unused)
        self.img_backbone_cfg, self.img_neck_cfg = cfg['img_backbone'], cfg['img_neck']
        self.train_cfg, self.test_cfg = train_cfg, cfg['test_cfg']
        if cfg['pts_backbone'] is not None:
            self.pts_backbone = build_backbone(cfg['pts_backbone'])
        if cfg['pts_neck'] is not None:
            self.pts_neck = build_neck(cfg['pts_neck'])
        if cfg['bbox_head'] is not None:
            head = dict(cfg['bbox_head'])
            if self.test_cfg is not None:
                # Assumption not checked against the reference source (srfdet.py:57-75), mmdet3d's MVX convention:
                route = self.test_cfg.get('pts', self.test_cfg)      # test_cfg.pts when present, else test_cfg itself
                head['test_cfg'] = dict(head.get('test_cfg') or {}, **route)
            self.bbox_head = build_head(head)
        self.use_graph = use_graph
        self._graphs = {}
        self.register_load_state_dict_pre_hook(self._drop_graphs_on_load)
        self.eval()

    @classmethod
    def from_config(cls, path_or_model):
        model = registry.load_config(path_or_model)['model'] if isinstance(path_or_model, str) else dict(path_or_model)
        model = dict(model)
        model.pop('type', None)
        return cls(**model)

    def reset_graphs(self):
        """Drop the captured graphs (they hold the weight buffers of the time of capture)."""
        self._graphs = {}

    def _drop_graphs_on_load(self, *args, **kwargs):
        self.reset_graphs()

    def _check_eval(self):
        if self.training:
            raise NotImplementedError('srfdet_b200 implements the inference path only (training mode is not supported)')

    # ------------------------------------------------------------------ checkpoints
    def load_checkpoint(self, path_or_state_dict, strict=True, trusted=False):
        """Load a reference checkpoint (file path or dict) by the reference's attribute names.  A file is read with
        torch.load(weights_only=True); trusted=True allows arbitrary pickled objects (mmcv checkpoints carry a `meta`
        with Python objects) -- only for files from a trusted source.  The state dict is ckpt['state_dict'] when
        present.  img_backbone.* / img_neck.* entries (modules not built here) are set aside, not errors.
        -> CheckpointKeys(missing_keys, unexpected_keys, set_aside_keys)."""
        ckpt = path_or_state_dict
        if isinstance(ckpt, (str, os.PathLike)):
            ckpt = torch.load(ckpt, map_location='cpu', weights_only=not trusted)
        sd = ckpt['state_dict'] if isinstance(ckpt, dict) and 'state_dict' in ckpt else ckpt
        sd = dict(sd)
        set_aside = sorted(k for k in sd if k.startswith(_IMAGE_PREFIXES))
        for k in set_aside:
            del sd[k]
        res = self.load_state_dict(sd, strict=strict)
        return CheckpointKeys(list(res.missing_keys), list(res.unexpected_keys), set_aside)

    # ------------------------------------------------------------------ device-resident forward
    @torch.no_grad()
    def voxelize_padded(self, points):
        """Hard voxelization + HardSimpleVFE of B clouds without a host read: every sample is voxelized into its own
        block of max_voxels rows, then srf_concat_counted_rows packs the valid rows in sample order.
        -> (voxel means (B * max_voxels, num_features), coors (B * max_voxels, 4) bzyx, count (1,) int32 device);
        rows past the count are unspecified."""
        assert isinstance(self.pts_voxel_encoder, HardSimpleVFE)
        blk = self.hard_voxel_blocks(points, want_mean=True)
        blk_coors, blk_mean, counts = blk['coors'], blk['mean'], blk['count']
        bs, mv, c = blk_mean.shape
        dev = blk_mean.device
        nf = self.pts_voxel_encoder.num_features
        coors = torch.empty((bs * mv, 4), dtype=torch.int32, device=dev)
        mean = torch.empty((bs * mv, nf), dtype=torch.float32, device=dev)
        total = torch.zeros((1,), dtype=torch.int32, device=dev)
        arrays = (L.Rows * 2)(L.Rows(blk_coors.data_ptr(), coors.data_ptr(), 4, 4, 4),
                              L.Rows(blk_mean.data_ptr(), mean.data_ptr(), c, nf, nf))
        L.check(L.load().srf_concat_counted_rows(L.ptr(counts), bs, mv, arrays, 2, L.ptr(total), L.stream_ptr()),
                'srf_concat_counted_rows')
        return mean, coors, total

    @torch.no_grad()
    def extract_point_features(self, points, precision=None):
        """As SRFDetPointPath; batches of hard-voxel HardSimpleVFE clouds also stay on the device (voxelize_padded)."""
        if len(points) > 1 and not self.is_dynamic and isinstance(self.pts_voxel_encoder, HardSimpleVFE):
            mean, coors, total = self.voxelize_padded(points)
            return self.pts_middle_encoder(mean, coors, len(points), num_voxels=total, precision=precision)
        return super().extract_point_features(points, precision)

    @torch.no_grad()
    def extract_pts_feat(self, points, precision=None):
        """points -> voxel encoder -> sparse encoder -> SECONDCustom -> FPN: list of BEV maps (B, C, H_l, W_l).
        Pillar configs: points -> pillar_rows -> SECONDCustom -> FPN."""
        from .bev_backbone import _tc_enc, nchw_to_rows
        precision = precision or registry.get_precision()
        if self.is_pillar:
            n = len(points)
            rows, h, w = self.pillar_rows(points, _tc_enc(precision))
        else:
            bev = self.extract_point_features(points, precision)
            n, _, h, w = bev.shape
            rows = nchw_to_rows(bev, _tc_enc(precision))
        feats = self.pts_backbone.forward_rows(rows, n, h, w, precision)
        return self.pts_neck.forward_rows(feats, n, precision)

    def extract_feat(self, points, img_feats=None, precision=None):
        """(img_feats, pts_feats) like srfdet.py:141-173; the image features are the caller's image-neck outputs."""
        return img_feats, self.extract_pts_feat(points, precision)

    def _check_inputs(self, points, img_feats, lidar2img):
        """Host-side checks of an infer call, before any device work."""
        self._check_eval()
        if not isinstance(points, (list, tuple)) or not points:
            raise ValueError('points must be a non-empty list of (N_i, C) CUDA tensors')
        if self.bbox_head.use_img:
            if img_feats is None or lidar2img is None:
                raise ValueError('this fusion config needs img_feats (the image-neck outputs, one (B, n_cam, C, H, W) map per '
                                 'level) and lidar2img (B, n_cam, 4, 4)')
            self._check_fusion_batch(len(points), img_feats, lidar2img)

    def _check_fusion_batch(self, n, img_feats, lidar2img):
        """n clouds need n samples of image maps and n camera sets (SURVEY.md §3.4: a batch of B fusion samples is B
        independent batch-1 calls).  One camera set for several clouds is the reference's own B > 1 case, which it does not
        define consistently (its RoI batch index and its feature flattening disagree): refused as such."""
        if not img_feats or any(f.dim() != 5 for f in img_feats):
            raise ValueError('img_feats: one (B, n_cam, C, H, W) image-neck map per level')
        batches, cams = {f.shape[0] for f in img_feats}, {f.shape[1] for f in img_feats}
        if len(batches) != 1 or len(cams) != 1:
            raise ValueError(f'every image level needs the same batch and camera count, got {[tuple(f.shape[:2]) for f in img_feats]}')
        mb, n_cam = batches.pop(), cams.pop()
        l2i = tuple(lidar2img.shape)
        if n > 1 and mb == 1 and l2i in ((n_cam, 4, 4), (1, n_cam, 4, 4)):
            raise NotImplementedError(
                f'the camera fusion branch has the reference\'s batch-size-1 semantics per sample: one camera set (image maps '
                f'of batch 1, lidar2img {l2i}) for {n} clouds is undefined there; pass each sample\'s maps as '
                f'({n}, {n_cam}, C, H, W) per level and lidar2img as ({n}, {n_cam}, 4, 4)')
        if mb != n:
            raise ValueError(f'image maps of batch {mb} for {n} clouds: the maps need one sample per cloud')
        if l2i != (n, n_cam, 4, 4) and not (n == 1 and l2i == (n_cam, 4, 4)):
            raise ValueError(f'lidar2img {l2i} does not match {n} sample(s) of {n_cam} cameras: pass ({n}, {n_cam}, 4, 4)')
        if getattr(self.bbox_head, 'with_dpg', False) and n > L.GEMV_MAX_ROWS:
            raise ValueError(f'{n} samples: the dynamic proposal generation projections (srf_gemv_f32) take at most '
                             f'{L.GEMV_MAX_ROWS} samples per call')

    @torch.no_grad()
    def _infer_eager(self, points, img_feats, lidar2img, precision):
        head = self.bbox_head
        img_feats, pyramid = self.extract_feat(points, img_feats, precision)
        logits, boxes = head(img_feats, pyramid, None, lidar2img=lidar2img, precision=precision)
        scores, dec = head.decode(logits, boxes)
        if head.device_nms:
            return head._nms_decoded(scores, dec)
        return scores, dec

    @torch.no_grad()
    def infer(self, points, img_feats=None, lidar2img=None, precision=None):
        """points: list of B (N_i, C) fp32 CUDA clouds; img_feats (fusion configs): per level (B, n_cam, C, H, W) image-neck
        maps, C = feat_channels_img (reduced by the head's img_convs) or hidden_dim; lidar2img (B, n_cam, 4, 4), or
        (n_cam, 4, 4) for one cloud.  Sample b is fused with its own maps img_feats[l][b] and projections lidar2img[b]: the
        B samples are B independent batch-1 calls of the reference (SURVEY.md §3.4).
        -> with the head's device NMS: boxes (B, max_per_img, dim-1), scores (B, max_per_img), labels (B, max_per_img)
        int32, counts (B,) int32 (SRFDetHead.nms_bboxes); otherwise the decoded (scores (B, P, #cls), boxes (B, P, dim-1)).
        No host synchronisation."""
        self._check_inputs(points, img_feats, lidar2img)
        precision = precision or registry.get_precision()
        if not self.use_graph:
            return self._infer_eager(points, img_feats, lidar2img, precision)
        key = (tuple(tuple(p.shape) for p in points), precision,
               None if img_feats is None else tuple((tuple(f.shape), f.stride()) for f in img_feats),
               None if lidar2img is None else tuple(lidar2img.shape))
        n, n_img = len(points), len(img_feats or [])

        def statics():
            return ([p.contiguous().clone() for p in points] + [torch.empty_like(f).copy_(f) for f in img_feats or []]
                    + [None if lidar2img is None else lidar2img.clone()])

        def run(*s):
            return self._infer_eager(list(s[:n]), list(s[n:n + n_img]) if img_feats is not None else None, s[-1], precision)
        return self._graph_call(key, statics, run, list(points) + list(img_feats or []) + [lidar2img])

    def _graph_call(self, key, statics, run, inputs):
        """run(*static inputs) captured into one CUDA graph per key (statics() makes the static copies of the inputs on
        first use) and replayed after `inputs` are copied into them; -> run's outputs, in graph-owned buffers."""
        g = self._graphs.get(key)
        if g is None:
            s_in = statics()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):          # warm-up off the capture: lazy kernel attributes, weight packing
                for _ in range(2):
                    run(*s_in)
            torch.cuda.current_stream().wait_stream(side)
            # the head memoises its img_convs outputs per input tensors: capture must record the convolutions themselves
            self.bbox_head._cache.pop('img_maps', None)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = run(*s_in)
            g = self._graphs[key] = (graph, s_in, out)
        graph, s_in, out = g
        for s, x in zip(s_in, inputs):
            if s is not None and s.data_ptr() != x.data_ptr():
                s.copy_(x, non_blocking=True)
        graph.replay()
        return out

    # ------------------------------------------------------------------ test-time augmentation
    def _check_aug(self):
        """Before any device work: TTA runs LiDAR-only configs with the head's device NMS."""
        self._check_eval()
        if self.bbox_head.use_img:
            raise NotImplementedError('test-time augmentation is built for LiDAR-only configs: camera fusion would need '
                                      'flipped images and lidar2img (DESIGN.md §1)')
        if not self.bbox_head.device_nms:
            raise NotImplementedError('test-time augmentation merges the views\' NMS results: it needs test_cfg.use_nms=True '
                                      'and the head\'s device NMS (no user nms_fn)')
        if self.bbox_head.test_cfg.get('max_num') is None:
            raise ValueError('test-time augmentation needs test_cfg.max_num (merge_aug_bboxes_3d keeps that many boxes)')

    def _merge_views(self, out, bs, views):
        """Per-view NMS outputs of a (bs * A)-cloud batch, sample-major -> merge_aug_bboxes_3d per sample."""
        from .nms import merge_aug_device
        boxes, scores, labels, counts = out
        a, m = len(views), boxes.shape[1]
        head, cfg = self.bbox_head, self.bbox_head.test_cfg
        # Assumptions not checked against the reference source (one line each):
        # SRFDet does not override mmdet3d's aug_test / aug_test_pts: views merged by merge_aug_bboxes_3d(test_cfg.pts).
        # LiDARInstance3DBoxes.flip (rc6): yaw = -yaw (horizontal), yaw = -yaw + pi (vertical), with_yaw boxes.
        # merge_aug_bboxes_3d uses nms_bev unless use_rotate_nms=False, like the head's get_bboxes.
        return merge_aug_device(boxes.view(bs, a, m, -1), scores.view(bs, a, m), labels.view(bs, a, m), counts.view(bs, a),
                                views, head.num_classes, cfg['nms_thr'], cfg.get('use_rotate_nms', True), cfg['max_num'])

    @torch.no_grad()
    def infer_aug(self, points, views, point_cloud_range=None, counts=None, precision=None):
        """Test-time augmentation of B clouds on the device: every cloud becomes its augmented views (srf_augment_points:
        scale, flips, then point_cloud_range -- the range filter of the test pipeline when it runs after the augmentation),
        all B x A views run as one batch through the detector with the head's device NMS, and srf_merge_aug_bev maps
        each view's boxes back and merges them per sample (mmdet3d merge_aug_bboxes_3d).  views: [(scale, horizontal flip,
        vertical flip)] (PointAugmentation.views); duplicates are dropped first (they would only repeat detections that
        the merge NMS removes again).  counts: (B,) int32 device numbers of valid rows (MultiSweepLoader), None: all rows.
        -> boxes (B, max_num, dim-1), scores (B, max_num), labels (B, max_num) int32, counts (B,) int32; rows past a count
        hold a zero box, score 0 and label -1.  No host synchronisation; use_graph=True: one graph per (shapes, views,
        range, precision)."""
        from .points import augment_points, distinct_views
        self._check_aug()
        self._check_inputs(points, None, None)
        views = distinct_views(views)
        if not 1 <= len(views) <= L.AUG_MAX_VIEWS:
            raise ValueError(f'{len(views)} distinct views: 1 to {L.AUG_MAX_VIEWS} are supported')
        precision = precision or registry.get_precision()
        rng = None if point_cloud_range is None else [float(v) for v in point_cloud_range]
        n = len(points)

        def run(*s):
            batch = []
            for i, p in enumerate(s[:n]):
                out, _ = augment_points(p, views, rng, None if s[n] is None else s[n][i:i + 1])
                batch += list(out)
            return self._merge_views(self._infer_eager(batch, None, None, precision), n, views)
        inputs = list(points) + [counts]
        if not self.use_graph:
            return run(*inputs)
        key = ('aug', tuple(tuple(p.shape) for p in points), tuple(views), None if rng is None else tuple(rng),
               counts is None, precision)
        return self._graph_call(key, lambda: [p.contiguous().clone() for p in points] + [None if counts is None else counts.clone()],
                                run, inputs)

    @torch.no_grad()
    def aug_test(self, points, img_metas, img=None, img_feats=None, rescale=False):
        """mmdet3d MVXTwoStageDetector.aug_test / aug_test_pts with SRFDet's head: points[a] / img_metas[a] are the
        already augmented clouds of augmentation a, one per sample, with their metas (pcd_scale_factor,
        pcd_horizontal_flip, pcd_vertical_flip).  All A x B clouds run as one batch, without dropping duplicates; the
        views' NMS results are merged per sample by srf_merge_aug_bev.  -> [dict(pts_bbox=dict(boxes_3d, scores_3d,
        labels_3d))] per sample, CPU tensors, boxes wrapped in box_type_3d when the metas give it; one read-back."""
        self._check_aug()
        if img is not None or img_feats is not None:
            raise NotImplementedError('test-time augmentation is built for LiDAR-only configs')
        a, bs = len(points), len(points[0])
        if any(len(p) != bs for p in points) or any(len(m) != bs for m in img_metas):
            raise ValueError('every augmentation needs the same number of clouds and metas')
        views = []
        for metas in img_metas:
            v = {(float(m.get('pcd_scale_factor', 1.0)), bool(m.get('pcd_horizontal_flip', False)),
                  bool(m.get('pcd_vertical_flip', False))) for m in metas}
            if len(v) != 1:
                raise ValueError(f'the samples of one augmentation have different flips / scales: {sorted(v)}')
            views.append(v.pop())
        clouds = [points[j][i] for i in range(bs) for j in range(a)]          # sample-major: the views of a sample together
        self._check_inputs(clouds, None, None)
        out = self._merge_views(self._infer_eager(clouds, None, None, registry.get_precision()), bs, views)
        res = self.bbox_head.format_nms(*out, [m for m in img_metas[0]])
        return [dict(pts_bbox=dict(boxes_3d=bx.to('cpu'), scores_3d=sc.cpu(), labels_3d=lb.cpu())) for bx, sc, lb in res]

    # ------------------------------------------------------------------ reference call contract
    @torch.no_grad()
    def simple_test(self, points, img_metas, img=None, img_feats=None, rescale=False):
        """srfdet.py:326-340 -> [dict(pts_bbox=dict(boxes_3d, scores_3d, labels_3d))] per sample, CPU tensors (mmdet3d
        bbox3d2result); boxes wrapped in img_metas[i]['box_type_3d'] when given.  One host read-back per call.
        Fusion configs: img_feats per level (B, n_cam, C, H, W); sample i is projected by img_metas[i]['lidar2img']."""
        self._check_eval()
        if img is not None and img_feats is None:
            raise ValueError('img= needs the image backbone and image neck, which are not built here '
                             f'(img_backbone: {(self.img_backbone_cfg or {}).get("type")}, img_neck: '
                             f'{(self.img_neck_cfg or {}).get("type")}): run them outside and pass their outputs as img_feats=')
        lidar2img = None
        if self.bbox_head.use_img and img_feats is not None:
            if len(img_metas) != len(points):
                raise ValueError(f'{len(points)} clouds with {len(img_metas)} img_metas: each sample needs its own meta')
            # one sample: its meta's (n_cam, 4, 4) as given; B samples: each from its own meta -> (B, n_cam, 4, 4)
            l2i = (np.asarray(img_metas[0]['lidar2img']) if len(img_metas) == 1
                   else np.stack([np.asarray(m['lidar2img']) for m in img_metas]))
            lidar2img = torch.as_tensor(l2i, dtype=torch.float32, device=points[0].device)
        out = self.infer(points, img_feats, lidar2img)
        head = self.bbox_head
        res = head.format_nms(*out, img_metas) if head.device_nms else head.select_decoded(*out, img_metas)
        return [dict(pts_bbox=dict(boxes_3d=bx.to('cpu'), scores_3d=sc.cpu(), labels_3d=lb.cpu())) for bx, sc, lb in res]

    def forward_test(self, points=None, img_metas=None, img=None, img_feats=None, **kwargs):
        """mmdet3d Base3DDetector.forward_test: points / img_metas (/ img) are lists over test-time augmentations."""
        for var, name in [(points, 'points'), (img_metas, 'img_metas')]:
            if not isinstance(var, list):
                raise TypeError(f'{name} must be a list, but got {type(var)}')
        if len(points) != len(img_metas):
            raise ValueError(f'num of augmentations ({len(points)}) != num of image meta ({len(img_metas)})')
        if len(points) > 1:
            return self.aug_test(points, img_metas, img=img, img_feats=img_feats, **kwargs)
        return self.simple_test(points[0], img_metas[0], img=None if img is None else img[0], img_feats=img_feats, **kwargs)

    def forward(self, return_loss=True, **kwargs):
        if return_loss:
            raise NotImplementedError('srfdet_b200 implements the inference path only: call forward(return_loss=False, ...)')
        return self.forward_test(**kwargs)


@DETECTORS.register_module(name='SRFDetWaymo')
class SRFDetWaymo(SRFDet):
    """SRFDetWaymo (srfdetwaymo.py:14-41): the SRFDet test path.
    Assumption not checked against the reference source: its simple_test returns the same per-sample
    dict(pts_bbox=...) nesting as SRFDet's."""
