"""Voxelization / DynamicScatter: the `mmdet3d.ops` symbols the reference imports
(detectors/srfdet.py:9, voxel_encoders/voxel_encoder.py:5), re-implemented over the
C ABI.  Same constructor arguments and forward contracts as mmcv 1.7.0."""
import ctypes

import torch
from torch import nn

from .. import _lib as L


def _ws(nbytes, device):
    return torch.empty((int(nbytes) + 255) // 256 * 256, dtype=torch.uint8, device=device)


class Voxelization(nn.Module):
    """mmcv.ops.Voxelization drop-in (call site detectors/srfdet.py:58,221,238).

    forward(points (N,C) f32 cuda):
      max_num_points == -1 -> coors (N,3) int32 (z,y,x), -1 rows when out of range
      else                 -> voxels (M,T,C), coors (M,3), num_points_per_voxel (M,)
    `max_voxels` may be an int or (train, test) like mmcv.
    """

    def __init__(self, voxel_size, point_cloud_range, max_num_points, max_voxels=20000, deterministic=True):
        super().__init__()
        self.voxel_size = list(voxel_size)
        self.point_cloud_range = list(point_cloud_range)
        self.max_num_points = max_num_points
        self.max_voxels = max_voxels if isinstance(max_voxels, (tuple, list)) else (max_voxels, max_voxels)
        self.deterministic = deterministic
        self.geom = L.make_geom(self.voxel_size, self.point_cloud_range)
        self.grid_size = [int(v) for v in self.geom.grid]

    def _max_voxels(self):
        return self.max_voxels[0] if self.training else self.max_voxels[1]

    def dynamic(self, points, batch_idx=-1):
        points = points.contiguous().float()
        n, c = points.shape
        coors = torch.empty((n, 3 if batch_idx < 0 else 4), dtype=torch.int32, device=points.device)
        L.check(L.load().srf_dynamic_voxelize(L.ptr(points), n, c, ctypes.byref(self.geom), batch_idx,
                                              L.ptr(coors), L.stream_ptr()), 'srf_dynamic_voxelize')
        return coors

    def hard_padded(self, points, batch_idx=-1, want_voxels=True, want_mean=False, want_p2v=False, out=None):
        """No host sync: outputs have max_voxels rows, the valid count stays on the device.
        -> dict(voxels, coors, num_points, mean, point2voxel, count).  out: caller-owned contiguous
        coors / num_points / mean / count tensors, and optionally voxels (one block of a batch buffer),
        written instead of new ones; their row count replaces max_voxels."""
        points = points.contiguous().float()
        n, c = points.shape
        dev = points.device
        mv, T = int(self._max_voxels()), int(self.max_num_points)
        if mv <= 0:
            mv = max(n, 1)
        if out is not None:
            mv = out['coors'].shape[0]
        lib = L.load()
        ws = _ws(lib.srf_hard_voxelize_ws_bytes(n, T, mv), dev)
        if out is None:
            out = dict(
                coors=torch.empty((mv, 3 if batch_idx < 0 else 4), dtype=torch.int32, device=dev),
                num_points=torch.empty((mv,), dtype=torch.int32, device=dev),
                mean=torch.empty((mv, c), dtype=torch.float32, device=dev) if want_mean else None,
                count=torch.zeros((1,), dtype=torch.int32, device=dev))
        voxels = out.get('voxels')
        if voxels is None and want_voxels:
            voxels = torch.empty((mv, T, c), dtype=torch.float32, device=dev)
        out = dict(out, voxels=voxels,
                   point2voxel=torch.empty((n,), dtype=torch.int32, device=dev) if want_p2v else None)
        L.check(lib.srf_hard_voxelize(L.ptr(points), n, c, ctypes.byref(self.geom), T, mv, batch_idx,
                                      L.ptr(out['voxels']), L.ptr(out['coors']), L.ptr(out['num_points']),
                                      L.ptr(out['mean']), L.ptr(out['point2voxel']), L.ptr(out['count']),
                                      L.ptr(ws), ws.numel(), L.stream_ptr()), 'srf_hard_voxelize')
        return out

    def forward(self, points):
        if self.max_num_points == -1:
            return self.dynamic(points)
        o = self.hard_padded(points)
        m = int(o['count'].item())  # the reference syncs here too (voxel_num readback in mmcv)
        return o['voxels'][:m], o['coors'][:m], o['num_points'][:m]

    def __repr__(self):
        return (f'{self.__class__.__name__}(voxel_size={self.voxel_size}, point_cloud_range='
                f'{self.point_cloud_range}, max_num_points={self.max_num_points}, max_voxels={self.max_voxels})')


class DynamicScatter(nn.Module):
    """mmcv.ops.DynamicScatter drop-in (voxel_encoder.py:82,99-102).

    forward(points (N,C), coors (N,3|4) int32) -> (voxel_feats (M,C), voxel_coors (M,3|4));
    rows with a negative coordinate are dropped, output sorted like at::unique_dim.
    mean reductions accumulate with float atomics (as mmcv does): order-nondeterministic
    in the last ulp; max is exact.
    """

    def __init__(self, voxel_size, point_cloud_range, average_points):
        super().__init__()
        self.voxel_size = list(voxel_size)
        self.point_cloud_range = list(point_cloud_range)
        self.average_points = average_points
        g = L.make_geom(self.voxel_size, self.point_cloud_range)
        self.grid_zyx = [int(g.grid[2]), int(g.grid[1]), int(g.grid[0])]

    def forward_padded(self, points, coors, batch_size=None, want_p2v=False):
        points = points.contiguous().float()
        coors = coors.contiguous().int()
        n, c = points.shape
        cd = coors.shape[1]
        dev = points.device
        if cd == 4:
            if batch_size is None:
                batch_size = int(coors[-1, 0].item()) + 1 if n else 1
            dims = [int(batch_size)] + self.grid_zyx
        else:
            dims = [1] + self.grid_zyx
        ncells = dims[0] * dims[1] * dims[2] * dims[3]
        lib = L.load()
        ws = _ws(lib.srf_scatter_ws_bytes(ncells, n, c), dev)
        feats = torch.empty((max(n, 1), c), dtype=torch.float32, device=dev)
        ocoors = torch.empty((max(n, 1), cd), dtype=torch.int32, device=dev)
        count = torch.zeros((1,), dtype=torch.int32, device=dev)
        p2v = torch.empty((n,), dtype=torch.int32, device=dev) if want_p2v else None
        L.check(lib.srf_dynamic_scatter(L.ptr(points), L.ptr(coors), n, c, cd, L.i4(dims),
                                        1 if self.average_points else 0, L.ptr(feats), L.ptr(ocoors),
                                        L.ptr(count), L.ptr(p2v), L.ptr(ws), ws.numel(), L.stream_ptr()),
                'srf_dynamic_scatter')
        return feats, ocoors, count, p2v

    def forward(self, points, coors):
        feats, ocoors, count, _ = self.forward_padded(points, coors)
        m = int(count.item())
        return feats[:m], ocoors[:m]
