"""Large LiDAR batches, host side (no GPU needed): the limits that remain are refused before any device work, with
messages that name them; srf_hard_voxelize_batch is in the ABI table; camera fusion keeps its 8-sample limit."""
import ctypes
import os

import pytest
import torch

from srfdet_b200 import _lib as L


def _det(golden_dir, name):
    from srfdet_b200.plugin import SRFDet, load_config
    det = SRFDet.from_config(load_config(os.path.join(golden_dir, 'configs', 'model', f'srfdet_{name}.py'))['model'])
    det.bbox_head.test_cfg['max_num'] = 500
    return det


def test_hard_voxelize_batch_in_abi_table():
    assert L.PROTOTYPES['srf_hard_voxelize_batch'][1][0] is ctypes.POINTER(ctypes.c_void_p)
    assert L.PROTOTYPES['srf_hard_voxelize_batch_ws_bytes'][0] is ctypes.c_size_t
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'srfdet_b200.h')).read()
    assert f'#define SRF_HV_BATCH_MAX {L.HV_BATCH_MAX}' in header
    assert not hasattr(L, 'GEMV_MAX_ROWS')


def test_batch_workspace_size():
    """The workspace query: one table per cloud, sized by the largest cloud; 0 for bad arguments."""
    lib = L.load()
    n = (ctypes.c_int32 * 3)(100, 0, 300000)
    one = lib.srf_hard_voxelize_ws_bytes(300000, 10, 160000)
    three = lib.srf_hard_voxelize_batch_ws_bytes(n, 3, 10, 160000)
    assert 2 * one < three < 3 * one + 2 ** 20
    assert lib.srf_hard_voxelize_batch_ws_bytes(n, 0, 10, 160000) == 0
    assert lib.srf_hard_voxelize_batch_ws_bytes((ctypes.c_int32 * 2)(5, -1), 2, 10, 160000) == 0


@pytest.mark.parametrize('name', ['nusc_L', 'pillar_nusc_L'])
def test_too_many_clouds_for_the_voxelizer(golden_dir, name):
    det = _det(golden_dir, name)
    with pytest.raises(ValueError, match=f'at most {L.HV_BATCH_MAX} clouds'):
        det.infer([torch.zeros(4, 5)] * (L.HV_BATCH_MAX + 1))
    with pytest.raises(ValueError, match=f'at most {L.HV_BATCH_MAX} clouds'):        # 79 clouds x 13 views
        det.infer_aug([torch.zeros(4, 5)] * 79, [(1.0 + 0.01 * i, False, False) for i in range(13)])


def test_tta_view_and_candidate_limits(golden_dir):
    """32 views per sample, and views x max_per_img <= 4096 merge candidates (nusc L: 300 rows, so 13 views)."""
    det = _det(golden_dir, 'nusc_L')
    assert det.bbox_head.test_cfg['max_per_img'] == 300
    pts = [torch.zeros(4, 5)]
    views = [(1.0 + 0.01 * i, False, False) for i in range(33)]
    with pytest.raises(ValueError, match='1 to 32'):
        det.infer_aug(pts, views)
    with pytest.raises(ValueError, match='at most 4096') as e:
        det.infer_aug(pts, views[:14])
    assert '14 views x 300 boxes' in str(e.value)
    metas = [[dict(pcd_scale_factor=s)] for s, _, _ in views]
    with pytest.raises(ValueError, match='1 to 32'):
        det.aug_test([pts] * 33, metas)
    with pytest.raises(ValueError, match='at most 4096'):
        det.aug_test([pts] * 14, metas[:14])


def test_voxelization_memory_check(golden_dir, monkeypatch):
    """A batch whose voxelization workspace and blocks do not fit in the free device memory is refused on the host."""
    det = _det(golden_dir, 'nusc_L')
    monkeypatch.setattr(torch.cuda, 'mem_get_info', lambda device=None: (2 ** 28, 180 * 2 ** 30))
    monkeypatch.setattr(torch.cuda, 'memory_reserved', lambda device=None: 0)
    monkeypatch.setattr(torch.cuda, 'memory_allocated', lambda device=None: 0)
    dev = torch.device('cuda', 0)
    det._check_voxel_batch([1000], 5, dev)                      # one small cloud fits in 256 MiB
    with pytest.raises(torch.cuda.OutOfMemoryError, match='32 clouds: hard voxelization needs'):
        det._check_voxel_batch([300000] * 32, 5, dev)


def test_fusion_still_refuses_nine_samples(golden_dir):
    """The camera-fusion path keeps its own limit of 8 samples per call (the LiDAR path has none)."""
    det = _det(golden_dir, 'nusc_LC')
    maps = [torch.zeros(9, 6, 128, 8 >> i, 8 >> i) for i in range(4)]
    with pytest.raises(ValueError, match='at most 8 samples'):
        det.infer([torch.zeros(4, 5)] * 9, img_feats=maps, lidar2img=torch.eye(4).expand(9, 6, 4, 4).clone())
