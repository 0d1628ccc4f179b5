"""The pillar config (PillarFeatureNetCustom + PointPillarsScatter + SECONDCustom + FPN + SRFDetHead) on the host (no
GPU): construction from the restated `model` config, the reference's state-dict names and the checkpoint round trip."""
import os

import pytest
import torch


def _cfg(golden_dir, kind='model'):
    return os.path.join(golden_dir, 'configs', kind, 'srfdet_pillar_nusc_L.py')


@pytest.mark.parametrize('kind', ['model', 'pipeline'])
def test_pillar_config_builds(golden_dir, kind):
    from srfdet_b200.plugin import (DETECTORS, FPN, PillarFeatureNetCustom, PointPillarsScatter, SECONDCustom, SRFDet,
                                    SRFDetHead, load_config)
    det = SRFDet.from_config(_cfg(golden_dir, kind))
    assert type(DETECTORS.build(load_config(_cfg(golden_dir, kind))['model'])) is SRFDet
    assert isinstance(det.pts_voxel_encoder, PillarFeatureNetCustom)
    assert isinstance(det.pts_middle_encoder, PointPillarsScatter)
    assert isinstance(det.pts_backbone, SECONDCustom) and isinstance(det.pts_neck, FPN) and isinstance(det.bbox_head, SRFDetHead)
    assert det.is_pillar and not det.is_dynamic and not det.training
    assert (det.pts_middle_encoder.ny, det.pts_middle_encoder.nx) == (512, 512)
    assert det.pts_voxel_layer.grid_size == [512, 512, 1]
    assert det.pts_voxel_layer.max_num_points == 20 and det.pts_voxel_layer._max_voxels() == 40000
    assert det.pts_voxel_encoder.in_channels == 11       # 5 raw + 3 cluster offsets + 3 pillar-centre offsets
    assert not det.bbox_head.use_img and det.bbox_head.use_nms


def test_pillar_state_dict_names(golden_dir):
    """Keys under the reference's attribute names; the DPG input is the (512 / (out_size_factor 2 * stride 8))^2 = 1024
    pixels of the pyramid's level the head pools."""
    from srfdet_b200.plugin import SRFDet
    sd = SRFDet.from_config(_cfg(golden_dir)).state_dict()
    assert tuple(sd['pts_voxel_encoder.pfn_layers.0.linear.weight'].shape) == (64, 11)
    assert tuple(sd['pts_voxel_encoder.pfn_layers.0.norm.running_var'].shape) == (64,)
    assert tuple(sd['pts_backbone.blocks.0.0.weight'].shape) == (64, 64, 3, 3)
    assert tuple(sd['pts_neck.lateral_convs.0.conv.weight'].shape) == (128, 64, 1, 1)
    assert sd['bbox_head.dpg_fc1_lidar.weight'].shape[1] == (512 // (2 * 8)) ** 2 == 1024
    assert not any(k.startswith('pts_middle_encoder.') for k in sd)      # PointPillarsScatter has no parameters
    assert all(k.startswith(('pts_voxel_encoder.', 'pts_backbone.', 'pts_neck.', 'bbox_head.')) for k in sd)


def test_pillar_checkpoint_round_trip(golden_dir, tmp_path):
    from srfdet_b200.plugin import SRFDet
    src = SRFDet.from_config(_cfg(golden_dir))
    g = torch.Generator().manual_seed(3)
    sd = {k: (v + torch.randn(v.shape, generator=g).to(v.dtype) if v.is_floating_point() else v.clone())
          for k, v in src.state_dict().items()}
    path = str(tmp_path / 'pillar.pth')
    torch.save({'state_dict': sd, 'meta': {'epoch': 20}}, path)
    det = SRFDet.from_config(_cfg(golden_dir))
    det._graphs['stale'] = object()
    res = det.load_checkpoint(path)
    assert res.missing_keys == [] and res.unexpected_keys == [] and res.set_aside_keys == []
    for k, v in det.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert det._graphs == {}
    broken = dict(sd)
    del broken['pts_voxel_encoder.pfn_layers.0.linear.weight']
    with pytest.raises(RuntimeError, match='pfn_layers.0.linear.weight'):
        SRFDet.from_config(_cfg(golden_dir)).load_checkpoint(broken)
