"""Test-time augmentation without a device: the MultiScaleFlipAug3D expansion of parse_test_augmentations against the
restated rc6 loops (aug_oracle), its rejections, the box mapping and the merge of the oracle itself, and the
argument checks that come before any device work."""
import itertools
import math
import os

import numpy as np
import pytest
import torch

import aug_oracle as O
import nms_oracle
from srfdet_b200.plugin import points as P
from srfdet_b200.plugin import registry

LOAD = dict(type='LoadPointsFromFile', load_dim=5, use_dim=5)
RANGE = dict(type='PointsRangeFilter', point_cloud_range=[-50, -50, -5, 50, 50, 3])
GRST = dict(type='GlobalRotScaleTrans', rot_range=[0, 0], scale_ratio_range=[0.95, 1.05], translation_std=[0, 0, 0])


def _pipeline(transforms, **aug):
    return [LOAD, dict(dict(type='MultiScaleFlipAug3D', img_scale=(1333, 800), transforms=transforms), **aug)]


@pytest.mark.parametrize('flip,h,v,sync_2d', list(itertools.product([False, True], repeat=4)))
@pytest.mark.parametrize('ratio', [1, [1.0], [0.95, 1.0, 1.05]])
def test_expansion_matches_rc6_loops(flip, h, v, sync_2d, ratio):
    aug = P.parse_test_augmentations(_pipeline([GRST, dict(type='RandomFlip3D', sync_2d=sync_2d), RANGE], pts_scale_ratio=ratio,
                                               flip=flip, pcd_horizontal_flip=h, pcd_vertical_flip=v))
    ref = O.expand_views(ratio, flip, h, v, sync_2d)
    assert aug.views == ref
    n_ratio = len(ratio) if isinstance(ratio, list) else 1
    assert len(aug.views) == n_ratio * (2 if flip else 1) * (2 if flip and h else 1) * (2 if flip and v else 1)
    assert P.distinct_views(aug.views) == list(dict.fromkeys(ref))
    assert aug.range_position == 'after' and aug.loader_steps.point_cloud_range is None
    assert aug.view_range == RANGE['point_cloud_range']


def test_double_flip_config():
    """The restated nusc_L TTA config: 8 views, 4 distinct, range filter after the augmentation, max_num in test_cfg."""
    d = os.path.join(os.path.dirname(__file__), 'golden', 'configs', 'pipeline')
    cfg = registry.load_config(os.path.join(d, 'srfdet_nusc_L_tta.py'))
    aug = P.parse_test_augmentations(cfg['test_pipeline'])
    assert len(aug.views) == 8 and P.distinct_views(aug.views) == [(1.0, h, v) for h in (False, True) for v in (False, True)]
    assert aug.views[4:] == aug.views[:4] and aug.augments
    assert aug.steps == P.parse_test_pipeline(registry.load_config(os.path.join(d, 'srfdet_nusc_L.py'))['test_pipeline'])
    assert cfg['model']['test_cfg']['pts']['max_num'] == 500
    with pytest.raises(NotImplementedError, match='MultiScaleFlipAug3D'):
        P.parse_test_pipeline(cfg['test_pipeline'])                      # the single-view parser keeps its contract


def test_duplicates_and_extra_loops():
    aug = P.parse_test_augmentations(_pipeline([dict(type='RandomFlip3D')], flip=True, pcd_horizontal_flip=True,
                                               flip_direction=['horizontal', 'vertical']))
    # sync_2d=True: horizontal follows `flip`; every view is repeated for each pcd flag and flip direction
    assert aug.views == O.expand_views(1, True, True, False, True, n_flip_direction=2)
    assert aug.views == [(1.0, False, False)] * 4 + [(1.0, True, False)] * 4
    aug = P.parse_test_augmentations(_pipeline([dict(type='RandomFlip3D')], img_scale=[(1333, 800), (1000, 600)]))
    assert aug.views == [(1.0, False, False)] * 2 and aug.augments


def test_range_position():
    assert P.parse_test_augmentations([LOAD, RANGE] + _pipeline([dict(type='RandomFlip3D')], flip=True)).range_position == 'before'
    aug = P.parse_test_augmentations(_pipeline([RANGE, dict(type='RandomFlip3D')], flip=True))
    assert aug.range_position == 'before' and aug.loader_steps.point_cloud_range == RANGE['point_cloud_range']
    assert aug.view_range is None
    assert P.parse_test_augmentations(_pipeline([dict(type='RandomFlip3D')], flip=True)).range_position is None
    plain = P.parse_test_augmentations([LOAD, RANGE])
    assert plain.views == [P.IDENTITY_VIEW] and not plain.augments


@pytest.mark.parametrize('pipeline,match', [
    (_pipeline([dict(type='RandomFlip3D'), RANGE], pts_scale_ratio=[0.95, 1.0]), 'GlobalRotScaleTrans'),
    (_pipeline([GRST, RANGE], flip=True), 'RandomFlip3D'),
    (_pipeline([dict(GRST, rot_range=[-0.1, 0.1]), dict(type='RandomFlip3D')], flip=True), 'rotation'),
    (_pipeline([dict(GRST, translation_std=[0.1, 0.1, 0.1])]), 'translation'),
    ([LOAD, dict(type='RandomFlip3D')], 'RandomFlip3D'),
    ([LOAD, GRST], 'GlobalRotScaleTrans'),
    (_pipeline([dict(type='RandomFlip3D')]) + _pipeline([dict(type='RandomFlip3D')]), 'one wrapper'),
    (_pipeline([dict(type='PointSample', num_points=100)]), 'PointSample'),
])
def test_rejections(pipeline, match):
    with pytest.raises(NotImplementedError, match=match):
        P.parse_test_augmentations(pipeline)


# ------------------------------------------------------------------------------------------ oracle geometry and merge
def _boxes(rng, n, dim=9, spread=30.0):
    b = np.zeros((n, dim), np.float32)
    b[:, :2] = rng.uniform(-spread, spread, (n, 2))
    b[:, 2] = rng.uniform(-2, 0, n)
    b[:, 3:6] = rng.uniform(0.5, 4.5, (n, 3))
    b[:, 6] = rng.uniform(-math.pi, math.pi, n)
    b[:, 7:] = rng.normal(0, 2, (n, dim - 7))
    return b


@pytest.mark.parametrize('scale', [1.0, 0.95, 1.05])
def test_mapping_back_round_trip(scale):
    """Augmenting a box (the forward flip and scale of its points) and mapping it back returns it: positions, extents
    and velocities within fp32 rounding of the scale, yaw up to the 2 pi of the vertical flip's + pi."""
    rng = np.random.default_rng(1)
    b = _boxes(rng, 200)
    for h, v in itertools.product([False, True], repeat=2):
        fwd = b.copy()
        fwd[:, :6] *= np.float32(scale)
        fwd[:, 7:] *= np.float32(scale)
        if h:
            fwd[:, 1::7] *= -1
            fwd[:, 6] = -fwd[:, 6]
        if v:
            fwd[:, 0::7] *= -1
            fwd[:, 6] = np.float32(np.pi) - fwd[:, 6]
        back = O.bbox3d_mapping_back(fwd, scale, h, v)
        keep = [0, 1, 2, 3, 4, 5, 7, 8]
        np.testing.assert_allclose(back[:, keep], b[:, keep], rtol=3e-7 if scale != 1 else 0, atol=1e-6 if scale != 1 else 0)
        dyaw = np.angle(np.exp(1j * (back[:, 6].astype(np.float64) - b[:, 6])))
        assert np.abs(dyaw).max() < 1e-6


def test_mapping_back_rules():
    """The rc6 rules themselves, on one row: y and vy (h), x and vx (v), yaw -yaw then -yaw + fl32(pi), scale last."""
    row = np.float32([[1, 2, 3, 4, 5, 6, 0.5, 7, 8]])
    np.testing.assert_array_equal(O.bbox3d_mapping_back(row, 1.0, True, False), np.float32([[1, -2, 3, 4, 5, 6, -0.5, 7, -8]]))
    np.testing.assert_array_equal(O.bbox3d_mapping_back(row, 1.0, False, True),
                                  np.float32([[-1, 2, 3, 4, 5, 6, np.float32(-0.5) + np.float32(np.pi), -7, 8]]))
    hv = O.bbox3d_mapping_back(row, 2.0, True, True)
    np.testing.assert_array_equal(hv, np.float32([[-0.5, -1, 1.5, 2, 2.5, 3, np.float32(0.5) + np.float32(np.pi), -3.5, -4]]))


@pytest.mark.parametrize('h,v', [(True, False), (False, True), (True, True)])
def test_flipped_footprint_is_mirrored(h, v):
    """The BEV footprint of a mapped-back box equals the mirror image of the detected box's footprint (flip) -- this pins
    position and extent; yaw +- pi gives the same footprint, so it cannot pin that."""
    rng = np.random.default_rng(2)
    for b in _boxes(rng, 50):
        back = O.bbox3d_mapping_back(b[None], 1.0, h, v)[0]
        mirrored = O.bev_footprint(b) * np.array([-1 if v else 1, -1 if h else 1])
        got = O.bev_footprint(back)
        d = np.abs(got[:, None, :] - mirrored[None, :, :]).max(-1)        # same corner set, any order
        assert d.min(1).max() < 1e-4 and d.min(0).max() < 1e-4


def _view_results(rng, n_views, n_cls, per_view=40):
    """Per-view detections of one scene seen through different views: shared objects jittered, distinct scores."""
    base = _boxes(rng, 30, spread=20.0)
    out = []
    for _ in range(n_views):
        idx = rng.integers(0, 30, per_view)
        b = base[idx].copy()
        b[:, :2] += rng.normal(0, 0.4, (per_view, 2)).astype(np.float32)
        out.append((b, rng.uniform(0.05, 0.95, per_view).astype(np.float32), rng.integers(0, n_cls, per_view)))
    return out


@pytest.mark.parametrize('n_cls', [1, 10])
def test_oracle_merge_duplicated_views_equal_distinct(n_cls):
    """Merging a duplicated view list equals merging its distinct views (first occurrence order): duplicates hold the
    same boxes, IoU 1 > thr, so the merge NMS removes them again.  Scenes without degenerate boxes."""
    rng = np.random.default_rng(3 + n_cls)
    views = [(1.0, False, False), (1.0, True, False), (0.95, False, True), (1.05, True, True)]
    res = _view_results(rng, 4, n_cls)
    order = [0, 1, 0, 2, 1, 3, 3, 2]
    full = O.merge_aug_bboxes_3d([res[i] for i in order], [views[i] for i in order], 0.4, 10 ** 6)
    distinct = O.merge_aug_bboxes_3d(res, views, 0.4, 10 ** 6)
    for a, b in zip(full[:3], distinct[:3]):
        np.testing.assert_array_equal(a, b)
    assert 0 < len(distinct[0]) < sum(len(r[0]) for r in res)
    cut = O.merge_aug_bboxes_3d(res, views, 0.4, 7)
    assert len(cut[0]) == 7 and (np.diff(cut[1]) <= 0).all()
    np.testing.assert_array_equal(cut[1], distinct[1][:7])


def test_missing_max_num_raises(golden_dir):
    from srfdet_b200.plugin import SRFDet
    det = SRFDet.from_config(os.path.join(golden_dir, 'configs', 'pipeline', 'srfdet_nusc_L.py'))
    pts = torch.zeros(4, 5)
    metas = [dict(pcd_horizontal_flip=False, pcd_vertical_flip=False, pcd_scale_factor=1.0)]
    with pytest.raises(ValueError, match='max_num'):
        det.forward_test(points=[[pts], [pts]], img_metas=[metas, metas])
    with pytest.raises(ValueError, match='max_num'):
        det.infer_aug([pts], [(1.0, False, False)])
    det.bbox_head.use_nms = False
    with pytest.raises(NotImplementedError, match='use_nms'):
        det.infer_aug([pts], [(1.0, False, False)])
