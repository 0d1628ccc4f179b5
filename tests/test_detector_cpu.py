"""SRFDet / SRFDetWaymo on the host (no GPU): construction from the full `model` configs, test_cfg routing, checkpoint
loading by the reference's attribute names and the test-time call contract's argument checks."""
import copy
import os

import pytest
import torch

CONFIGS = ['nusc_LC', 'nusc_L', 'waymo_L', 'kitti_L']
PREFIXES = ('pts_voxel_encoder.', 'pts_middle_encoder.', 'pts_backbone.', 'pts_neck.', 'bbox_head.')


def _model(golden_dir, name):
    from srfdet_b200.plugin import load_config
    return load_config(os.path.join(golden_dir, 'configs', 'model', f'srfdet_{name}.py'))['model']


@pytest.mark.parametrize('name', CONFIGS)
def test_detector_builds_from_full_config(golden_dir, name):
    from srfdet_b200.plugin import (DETECTORS, FPN, SECONDCustom, SparseEncoderCustom, SRFDet, SRFDetHead, SRFDetPointPath,
                                    SRFDetWaymo)
    model = _model(golden_dir, name)
    det = SRFDet.from_config(os.path.join(golden_dir, 'configs', 'model', f'srfdet_{name}.py'))
    via_registry = DETECTORS.build(model)
    assert type(via_registry) is (SRFDetWaymo if name.startswith('waymo') else SRFDet)
    assert isinstance(via_registry, SRFDetPointPath)
    assert isinstance(det.pts_middle_encoder, SparseEncoderCustom) and isinstance(det.pts_backbone, SECONDCustom)
    assert isinstance(det.pts_neck, FPN) and isinstance(det.bbox_head, SRFDetHead)
    assert not det.training
    assert [n for n, _ in det.named_children()] == ['pts_voxel_layer', 'pts_voxel_encoder', 'pts_middle_encoder',
                                                     'pts_backbone', 'pts_neck', 'bbox_head']
    keys = list(det.state_dict())
    assert keys and all(k.startswith(PREFIXES) for k in keys)
    for p in ('pts_middle_encoder.', 'pts_backbone.', 'pts_neck.', 'bbox_head.'):
        assert any(k.startswith(p) for k in keys), p
    # each sub-tree has exactly the keys of the module built on its own from the same config
    for attr, build in [('pts_backbone', 'build_backbone'), ('pts_neck', 'build_neck'), ('bbox_head', 'build_head')]:
        from srfdet_b200.plugin import registry
        ref = getattr(registry, build)(model[attr])
        assert sorted(k[len(attr) + 1:] for k in keys if k.startswith(attr + '.')) == sorted(ref.state_dict())
    assert det.bbox_head.use_img == (name == 'nusc_LC')
    if name == 'nusc_LC':
        assert hasattr(det.bbox_head, 'img_convs')
        assert det.img_backbone_cfg == dict(type='ImageBackbonePlaceholder')        # kept, init_cfg dropped, not built
        assert det.img_neck_cfg == dict(type='ImageNeckPlaceholder')
        assert not any(k.startswith(('img_backbone', 'img_neck')) for k in keys)


@pytest.mark.parametrize('name', ['nusc_L', 'kitti_L'])
def test_point_path_only_config_matches_point_path(golden_dir, name):
    from srfdet_b200.plugin import SRFDet, SRFDetPointPath
    model = _model(golden_dir, name)
    point = {k: model[k] for k in ('pts_voxel_layer', 'pts_voxel_encoder', 'pts_middle_encoder')}
    a, b = SRFDet(**copy.deepcopy(point)), SRFDetPointPath(**copy.deepcopy(point))
    assert list(a.state_dict()) == list(b.state_dict())
    assert [(n, type(m)) for n, m in a.named_modules()][1:] == [(n, type(m)) for n, m in b.named_modules()][1:]


def test_init_cfg_and_pretrained_dropped_at_every_level(golden_dir):
    from srfdet_b200.plugin import SRFDet
    model = _model(golden_dir, 'kitti_L')
    model['pretrained'] = 'ckpt.pth'
    model['pts_middle_encoder']['init_cfg'] = dict(type='Pretrained', checkpoint='enc.pth')
    model['pts_backbone']['init_cfg'] = dict(type='Kaiming')
    model['pts_neck']['init_cfg'] = dict(type='Xavier')
    model['bbox_head']['init_cfg'] = dict(type='Normal')
    model['bbox_head']['pretrained'] = 'head.pth'
    det = SRFDet.from_config(model)
    assert det.pts_middle_encoder.init_cfg is None
    assert 'pretrained' not in det.unused_cfg


@pytest.mark.parametrize('form', ['pts', 'flat'])
def test_test_cfg_routing(golden_dir, form):
    from srfdet_b200.plugin import SRFDet
    model = _model(golden_dir, 'nusc_L')
    pts_cfg = model['test_cfg']['pts']
    model['bbox_head']['test_cfg'] = dict(max_per_img=50, score_thr=0.1, use_nms=False)     # merged under the model-level one
    model['test_cfg'] = dict(pts=pts_cfg) if form == 'pts' else dict(pts_cfg)
    head = SRFDet.from_config(model).bbox_head
    assert head.test_cfg == dict(score_thr=0.1, **pts_cfg)
    assert head.use_nms and head.test_cfg['max_per_img'] == 300 and head.test_cfg['nms_thr'] == 0.4
    model['test_cfg'] = None
    head = SRFDet.from_config(model).bbox_head
    assert head.test_cfg == dict(max_per_img=50, score_thr=0.1, use_nms=False) and not head.use_nms


def _perturbed(det, seed):
    g = torch.Generator().manual_seed(seed)
    return {k: (v + torch.randn(v.shape, generator=g).to(v.dtype) if v.is_floating_point() else v.clone())
            for k, v in det.state_dict().items()}


def test_load_checkpoint_round_trip(golden_dir, tmp_path):
    from srfdet_b200.plugin import SRFDet
    det = SRFDet.from_config(_model(golden_dir, 'nusc_LC'))
    sd = _perturbed(det, 0)
    full = dict(sd, **{'img_backbone.stem.weight': torch.zeros(3), 'img_neck.lateral.0.weight': torch.zeros(2)})
    path = str(tmp_path / 'epoch_3.pth')
    torch.save({'state_dict': full, 'meta': {'epoch': 3, 'CLASSES': ('car', 'truck'), 'mmdet3d_version': '1.0.0rc6'}}, path)
    fresh = SRFDet.from_config(_model(golden_dir, 'nusc_LC'))
    res = fresh.load_checkpoint(path)
    assert res.missing_keys == [] and res.unexpected_keys == []
    assert res.set_aside_keys == ['img_backbone.stem.weight', 'img_neck.lateral.0.weight']
    for k, v in fresh.state_dict().items():
        assert torch.equal(v, sd[k]), k
    # a plain state dict (no 'state_dict' wrapper) loads too
    assert SRFDet.from_config(_model(golden_dir, 'nusc_LC')).load_checkpoint(sd).set_aside_keys == []
    # a genuinely missing head key still fails with strict=True, and is reported with strict=False
    broken = dict(full)
    del broken['bbox_head.dpg_fc1_lidar.weight']
    with pytest.raises(RuntimeError, match='dpg_fc1_lidar'):
        SRFDet.from_config(_model(golden_dir, 'nusc_LC')).load_checkpoint(broken)
    res = SRFDet.from_config(_model(golden_dir, 'nusc_LC')).load_checkpoint(broken, strict=False)
    assert res.missing_keys == ['bbox_head.dpg_fc1_lidar.weight']


def test_load_checkpoint_untrusted_file_rejects_pickled_objects(golden_dir, tmp_path):
    from srfdet_b200.plugin import SRFDet
    det = SRFDet.from_config(_model(golden_dir, 'kitti_L'))
    path = str(tmp_path / 'ckpt.pth')
    torch.save({'state_dict': det.state_dict(), 'meta': {'config': _Opaque()}}, path)
    with pytest.raises(Exception):
        det.load_checkpoint(path)
    assert det.load_checkpoint(path, trusted=True).missing_keys == []


class _Opaque:
    pass


def test_weight_caches_follow_detector_load_checkpoint(golden_dir):
    """The packed-weight caches of the encoders and the head are keyed on (data_ptr, version) of their sources, so a
    checkpoint loaded at the detector level invalidates them (as tests/test_plugin_cpu.py checks one level down)."""
    from srfdet_b200.plugin import SRFDet
    from srfdet_b200.plugin.head import _cached
    det = SRFDet.from_config(_model(golden_dir, 'waymo_L'))
    enc0, vfe0 = det.pts_middle_encoder._weights_version(), det.pts_voxel_encoder._weights_version()
    fc = det.bbox_head.dpg_fc1_lidar
    cache, calls = {}, []
    make = lambda: calls.append(1) or len(calls)
    assert _cached(cache, 'k', (fc.weight,), make) == 1 and _cached(cache, 'k', (fc.weight,), make) == 1
    det._graphs['stale'] = object()
    det.load_checkpoint({'state_dict': _perturbed(det, 1)})
    assert det.pts_middle_encoder._weights_version() != enc0 and det.pts_voxel_encoder._weights_version() != vfe0
    assert _cached(cache, 'k', (fc.weight,), make) == 2
    assert det._graphs == {}          # captured graphs bake in weight buffers: dropped on load


def test_test_time_contract_argument_checks(golden_dir):
    from srfdet_b200.plugin import SRFDet
    det = SRFDet.from_config(_model(golden_dir, 'nusc_LC'))
    pts = torch.zeros(4, 5)
    metas = [dict(lidar2img=torch.eye(4).repeat(6, 1, 1).numpy())]
    with pytest.raises(NotImplementedError, match='augmentation'):
        det.forward_test(points=[[pts], [pts]], img_metas=[metas, metas])
    with pytest.raises(NotImplementedError, match='augmentation'):
        det(return_loss=False, points=[[pts], [pts]], img_metas=[metas, metas])
    with pytest.raises(ValueError, match='img_feats') as e:
        det.forward_test(points=[[pts]], img_metas=[metas], img=[torch.zeros(1, 6, 3, 32, 32)])
    assert 'ImageBackbonePlaceholder' in str(e.value) and 'image neck' in str(e.value)
    with pytest.raises(ValueError, match='img_feats'):
        det.simple_test([pts], metas)                            # fusion config without image features
    with pytest.raises(NotImplementedError):
        det(points=[[pts]], img_metas=[metas])                   # return_loss=True: training
    det.train()
    with pytest.raises(NotImplementedError, match='inference'):
        det.simple_test([pts], metas)
    with pytest.raises(NotImplementedError, match='inference'):
        det.infer([pts])
