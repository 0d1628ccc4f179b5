"""Pillar path of the srfdet_pillar_* configs (SURVEY.md 8f rank 4):
PillarFeatureNetCustom (mmdet3d_plugin/models/voxel_encoders/pillar_encoder_custom.py:13-161,
PFNLayer voxel_encoders/utils.py:85-147) and mmdet3d's PointPillarsScatter
(cfg configs/nus/srfdet_pillar_nusc_L.py:37-54), same registry names / constructor arguments /
state-dict keys, forward on the fused `srf_pillar_vfe` / `srf_pillars_scatter` kernels."""
import torch
from torch import nn

from .. import _lib as L
from .registry import MIDDLE_ENCODERS, VOXEL_ENCODERS, build_norm_layer
from .voxel_encoder import fold_bn


class PFNLayer(nn.Module):
    """Parameter holder with the reference's names (`linear.weight`, `norm.*`)."""

    def __init__(self, in_channels, out_channels, norm_cfg=dict(type='BN1d', eps=1e-3, momentum=0.01), last_layer=False,
                 mode='max'):
        super().__init__()
        assert mode in ('max', 'avg')
        self.last_vfe = last_layer
        if not last_layer:
            out_channels = out_channels // 2
        self.units = out_channels
        self.norm = build_norm_layer(norm_cfg, self.units)[1]
        self.linear = nn.Linear(in_channels, self.units, bias=False)
        self.mode = mode


@VOXEL_ENCODERS.register_module()
class PillarFeatureNetCustom(nn.Module):
    def __init__(self, in_channels=4, feat_channels=(64,), with_distance=False, with_cluster_center=True,
                 with_voxel_center=True, voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1),
                 norm_cfg=dict(type='BN1d', eps=1e-3, momentum=0.01), mode='max', legacy=True, init_cfg=None):
        super().__init__()
        assert len(feat_channels) > 0
        self.legacy = legacy
        self.raw_in_channels = in_channels
        in_channels += 3 * int(with_cluster_center) + 3 * int(with_voxel_center) + int(with_distance)
        self._with_distance, self._with_cluster_center, self._with_voxel_center = with_distance, with_cluster_center, with_voxel_center
        self.in_channels = in_channels
        chans = [in_channels] + list(feat_channels)
        self.pfn_layers = nn.ModuleList([PFNLayer(chans[i], chans[i + 1], norm_cfg=norm_cfg, last_layer=i == len(chans) - 2, mode=mode)
                                         for i in range(len(chans) - 1)])
        self.mode = mode
        self.vx, self.vy, self.vz = voxel_size
        self.x_offset = self.vx / 2 + point_cloud_range[0]
        self.y_offset = self.vy / 2 + point_cloud_range[1]
        self.z_offset = self.vz / 2 + point_cloud_range[2]
        self.point_cloud_range = point_cloud_range
        self._folded = None

    def _fold(self, device):
        layer = self.pfn_layers[0]
        src = [layer.linear.weight] + list(layer.norm.parameters()) + list(layer.norm.buffers())
        ver = tuple((t.data_ptr(), t._version) for t in src)
        if self._folded is None or self._folded[0] != (ver, str(device)):
            w, b = fold_bn(layer.linear.weight, layer.norm)
            self._folded = ((ver, str(device)), w.to(device).contiguous(), b.to(device).contiguous())
        return self._folded[1], self._folded[2]

    def _kernel_args(self, device):
        """(folded weight, folded bias, flags word) of the fused PFN kernels."""
        if self.training:
            raise NotImplementedError('srfdet_b200 implements the inference path only')
        if len(self.pfn_layers) != 1:
            raise NotImplementedError('the fused kernel implements the single-PFNLayer form every reference config uses')
        w, b = self._fold(device)
        flags = int(self._with_cluster_center) | (int(self._with_voxel_center) << 1) | (int(self._with_distance) << 2) \
            | (int(bool(self.legacy)) << 3) | (int(self.mode == 'avg') << 4)
        return w, b, flags

    def forward(self, features, num_points, coors, num_voxels=None):
        """features (N, T, C) zero-padded pillars, num_points (N,), coors (N,4) (b,z,y,x) -> (N, C_out).
        num_voxels: optional (1,) int32 device count of valid rows (no-sync path)."""
        features = features.contiguous().float()
        n, t, c = features.shape
        layer = self.pfn_layers[0]
        w, b, flags = self._kernel_args(features.device)
        out = torch.empty((n, layer.units), dtype=torch.float32, device=features.device)
        L.check(L.load().srf_pillar_vfe(L.ptr(features), L.ptr(num_points.contiguous().int()), L.ptr(coors.contiguous().int()), n,
                                        L.ptr(num_voxels), t, c, L.ptr(w), L.ptr(b), layer.units, L.f3([self.vx, self.vy, self.vz]),
                                        L.f3([self.x_offset, self.y_offset, self.z_offset]), flags, L.ptr(out), L.stream_ptr()),
                'srf_pillar_vfe')
        return out

    def encode_rows(self, voxels, num_points, coors, counts, ny, nx, enc):
        """This module followed by PointPillarsScatter and the NCHW -> pixel-row encoding of the dense backbone, in one
        kernel (srf_pillar_encode_rows) and without a canvas.  voxels (B, M, T, C), num_points (B, M), coors (B, M, 4)
        int32: per-sample blocks of hard voxelization; counts (B,) int32 device counts of valid rows per block.
        -> rows ((B*ny*nx + 127) // 128 * 128, enc_width(enc, C_out)) in encoding enc: row (b*ny + y)*nx + x holds the
        features of sample b's pillar at (y, x), empty cells are zero; the rows past B*ny*nx are unspecified padding."""
        bs, m, t, c = voxels.shape
        layer = self.pfn_layers[0]
        w, b, flags = self._kernel_args(voxels.device)
        rows = torch.empty(((bs * ny * nx + 127) // 128 * 128, L.enc_width(enc, layer.units)), dtype=L.enc_torch_dtype(enc),
                           device=voxels.device)
        L.check(L.load().srf_pillar_encode_rows(L.ptr(voxels), L.ptr(num_points), L.ptr(coors), L.ptr(counts), bs, m, t, c,
                                                L.ptr(w), L.ptr(b), layer.units, L.f3([self.vx, self.vy, self.vz]),
                                                L.f3([self.x_offset, self.y_offset, self.z_offset]), flags, ny, nx, enc,
                                                L.ptr(rows), L.stream_ptr()), 'srf_pillar_encode_rows')
        return rows


@MIDDLE_ENCODERS.register_module()
class PointPillarsScatter(nn.Module):
    """[3P] mmdet3d PointPillarsScatter: (N, C) pillar features + (N,4) (b,z,y,x) -> (B, C, ny, nx) canvas."""

    def __init__(self, in_channels, output_shape):
        super().__init__()
        self.in_channels = in_channels
        self.ny, self.nx = int(output_shape[0]), int(output_shape[1])
        self.channels_last = False   # True: emit a torch.channels_last canvas for the dense backbone kernels

    def forward(self, voxel_features, coors, batch_size=None, num_voxels=None):
        voxel_features = voxel_features.contiguous().float()
        coors = coors.contiguous().int()
        n, c = voxel_features.shape
        if batch_size is None:
            batch_size = int(coors[:, 0].max().item()) + 1 if n else 1
        canvas = torch.empty((batch_size, c, self.ny, self.nx), dtype=torch.float32, device=voxel_features.device,
                             memory_format=torch.channels_last if self.channels_last else torch.contiguous_format).zero_()
        return self.scatter_into(canvas, voxel_features, coors, num_voxels)

    def scatter_into(self, canvas, voxel_features, coors, num_voxels=None):
        """forward into a caller-owned zeroed canvas (B, C, ny, nx) (torch.channels_last when self.channels_last): lets a
        batch voxelized in per-sample blocks be scattered block by block, each with its own device count."""
        n, c = voxel_features.shape
        L.check(L.load().srf_pillars_scatter(L.ptr(voxel_features), L.ptr(coors), n, L.ptr(num_voxels), c, self.ny, self.nx,
                                             int(self.channels_last), canvas.data_ptr(), L.stream_ptr()), 'srf_pillars_scatter')
        return canvas
