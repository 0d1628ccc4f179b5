"""Multi-sweep point input without a GPU: the numpy restatement against the literal rc6 transcription, the sweep choice,
test-pipeline parsing, the restricted nuScenes infos reader and the loader's host-side checks (plugin/points.py)."""
import os
import pickle

import numpy as np
import pytest

import sweep_oracle as O
from srfdet_b200.plugin import points as P
from srfdet_b200.plugin import registry

NUSC_SWEEPS = dict(sweeps_num=10, load_dim=5, use_dim=[0, 1, 2, 3, 4], pad_empty_sweeps=True, remove_close=True)


def _pipeline_cfg(golden_dir, name):
    return os.path.join(golden_dir, 'configs', 'pipeline', f'srfdet_{name}.py')


@pytest.mark.parametrize('remove_close', [False, True])
@pytest.mark.parametrize('n_sweeps', [[], [900, 0, 700], [300] * 12])
@pytest.mark.parametrize('pad', [False, True])
def test_oracle_equals_literal(remove_close, n_sweeps, pad):
    """Same kept set and order; values within 1 float32 ulp (BLAS may sum the rotation in another order)."""
    rng = np.random.default_rng(len(n_sweeps) * 4 + 2 * remove_close + pad)
    sample = O.make_sample(rng, 1000, n_sweeps)
    sw = dict(NUSC_SWEEPS, remove_close=remove_close, pad_empty_sweeps=pad, test_mode=True)
    got = O.merge(sample, 5, 5, sw, O.NUSC_RANGE, choices=P.choose_sweeps(len(n_sweeps), 10, True))
    ref = O.literal_pipeline(sample, 5, 5, sw, O.NUSC_RANGE)
    assert got.shape == ref.shape and got.shape[0] > 500
    np.testing.assert_array_equal(got[:, 3:], ref[:, 3:])
    np.testing.assert_array_max_ulp(got[:, :3], ref[:, :3], maxulp=1)


def test_edge_points_follow_the_reference():
    """|x| or |y| exactly 1 survives remove_close (strict <); points exactly on a range face are removed (strict <)."""
    e = O.edge_points()
    kept = O.remove_close(e)
    assert not any((abs(p[0]) < 1 and abs(p[1]) < 1) for p in kept) and len(kept) == len(e) - 2
    inside = O.range_filter(e, O.NUSC_RANGE)
    lo, hi = np.float32(O.NUSC_RANGE[:3]), np.float32(O.NUSC_RANGE[3:])
    assert len(inside) == len(e) - 6
    assert ((inside[:, :3] > lo) & (inside[:, :3] < hi)).all()


def test_choose_sweeps_matches_reference():
    """All sweeps when there are at most sweeps_num; the first sweeps_num in test_mode; otherwise the reference's draw
    from numpy's global generator."""
    assert P.choose_sweeps(3, 10, False) == [0, 1, 2] and P.choose_sweeps(0, 10, False) == []
    assert P.choose_sweeps(13, 10, True) == list(range(10))
    np.random.seed(7)
    got = P.choose_sweeps(13, 10, False)
    np.random.seed(7)
    assert got == list(np.random.choice(13, 10, replace=False)) and len(set(got)) == 10 and got != list(range(10))
    # the literal transcription draws the same sweeps
    rng = np.random.default_rng(3)
    sample = O.make_sample(rng, 200, [50] * 13, edges=False)
    sw = dict(NUSC_SWEEPS, remove_close=False, pad_empty_sweeps=False)
    np.random.seed(11)
    choices = P.choose_sweeps(13, 10, False)
    np.random.seed(11)
    ref = O.literal_pipeline(sample, 5, 5, sw, None)
    got = O.merge(sample, 5, 5, sw, None, choices=choices)
    np.testing.assert_array_equal(got[:, 3:], ref[:, 3:])


def test_pad_empty_sweeps_repeats_key_frame():
    rng = np.random.default_rng(4)
    sample = O.make_sample(rng, 400, [])
    for close in (False, True):
        got = O.literal_pipeline(sample, 5, 5, dict(NUSC_SWEEPS, remove_close=close), None)
        key = O.load(sample['lidar_path'], 5)
        rep = O.remove_close(key) if close else key
        assert got.shape[0] == key.shape[0] + 10 * rep.shape[0]
        assert (got[:, 4] == 0).all()


def test_parse_reference_pipelines(golden_dir):
    st = P.parse_test_pipeline(registry.load_config(_pipeline_cfg(golden_dir, 'nusc_L'))['test_pipeline'])
    assert st.load_dim == 5 and st.use_dim == [0, 1, 2, 3, 4] and st.point_cloud_range == O.NUSC_RANGE
    assert st.sweeps == dict(NUSC_SWEEPS, test_mode=False)
    st = P.parse_test_pipeline(registry.load_config(_pipeline_cfg(golden_dir, 'waymo_L'))['test_pipeline'])
    assert st.load_dim == 6 and st.use_dim == [0, 1, 2, 3, 4] and st.sweeps is None
    assert st.point_cloud_range == [-76.8, -76.8, -2, 76.8, 76.8, 4]


def _aug(*transforms, **kw):
    return [dict(type='LoadPointsFromFile', load_dim=5, use_dim=5),
            dict(type='MultiScaleFlipAug3D', img_scale=(1333, 800), pts_scale_ratio=kw.get('ratio', 1),
                 flip=kw.get('flip', False), transforms=list(transforms))]


@pytest.mark.parametrize('pipeline, name', [
    (_aug(dict(type='GlobalRotScaleTrans', rot_range=[-0.1, 0.1], scale_ratio_range=[1, 1], translation_std=[0, 0, 0])),
     'GlobalRotScaleTrans'),
    (_aug(dict(type='GlobalRotScaleTrans', rot_range=[0, 0], scale_ratio_range=[0.95, 1.05])), 'GlobalRotScaleTrans'),
    (_aug(dict(type='GlobalRotScaleTrans')), 'GlobalRotScaleTrans'),
    (_aug(dict(type='RandomFlip3D'), flip=True), 'MultiScaleFlipAug3D'),
    (_aug(ratio=[0.9, 1.0]), 'MultiScaleFlipAug3D'),
    (_aug(dict(type='PointShuffle')), 'PointShuffle'),
    ([dict(type='LoadPointsFromFile', load_dim=5, use_dim=5), dict(type='RandomFlip3D', flip_ratio_bev_horizontal=0.5)],
     'RandomFlip3D'),
])
def test_non_identity_augmentation_raises(pipeline, name):
    with pytest.raises(NotImplementedError, match=name):
        P.parse_test_pipeline(pipeline)


def test_parse_ignores_image_steps_and_checks_columns():
    st = P.parse_test_pipeline([dict(type='LoadPointsFromFile', load_dim=5, use_dim=5),
                                dict(type='LoadMultiViewImageFromFiles', to_float32=True),
                                dict(type='LoadPointsFromMultiSweeps', sweeps_num=3, use_dim=[0, 1, 2, 4]),
                                dict(type='NormalizeMultiviewImage', mean=[0, 0, 0], std=[1, 1, 1]),
                                dict(type='Collect3D', keys=['points', 'img'])])
    assert st.sweeps['sweeps_num'] == 3 and st.sweeps['use_dim'] == [0, 1, 2, 4] and st.point_cloud_range is None
    with pytest.raises(ValueError, match='concatenates'):
        P.parse_test_pipeline([dict(type='LoadPointsFromFile', load_dim=5, use_dim=4),
                               dict(type='LoadPointsFromMultiSweeps', sweeps_num=3)])
    with pytest.raises(ValueError, match='LoadPointsFromFile'):
        P.parse_test_pipeline([dict(type='LoadPointsFromMultiSweeps', sweeps_num=3)])


def test_loader_needs_test_pipeline(golden_dir):
    cfg = os.path.join(golden_dir, 'configs', 'model', 'srfdet_nusc_L.py')
    with pytest.raises(ValueError, match='test_pipeline'):
        P.MultiSweepLoader.from_config(cfg)


# ------------------------------------------------------------------------------------- nuScenes infos
def _infos(tmp_path, protocol):
    rng = np.random.default_rng(0)
    info = dict(lidar_path='./data/nuscenes/samples/LIDAR_TOP/a.pcd.bin', token='t0', timestamp=1533151603547590,
                lidar2ego_rotation=[1.0, 0.0, 0.0, 0.0], cams=dict(CAM_FRONT=dict(data_path='x.jpg')),
                sweeps=[dict(data_path='./data/nuscenes/sweeps/LIDAR_TOP/b.pcd.bin', type='lidar',
                             sensor2lidar_rotation=O.random_rotation(rng), sensor2lidar_translation=rng.normal(size=3),
                             timestamp=1533151603497590)],
                gt_boxes=np.zeros((0, 7), np.float32), num_lidar_pts=np.array([3, 4]), valid_flag=np.array([True, False]),
                score=np.float64(0.5))
    path = tmp_path / f'infos_p{protocol}.pkl'
    with open(path, 'wb') as f:
        pickle.dump(dict(infos=[info], metadata=dict(version='v1.0-trainval')), f, protocol=protocol)
    return str(path), info


@pytest.mark.parametrize('protocol', [2, 4])
def test_info_reader(tmp_path, protocol):
    path, info = _infos(tmp_path, protocol)
    got = P.load_nuscenes_infos(path)
    assert len(got) == 1 and got[0]['lidar_path'] == info['lidar_path'] and got[0]['timestamp'] == info['timestamp']
    s, r = got[0]['sweeps'][0], info['sweeps'][0]
    np.testing.assert_array_equal(s['sensor2lidar_rotation'], r['sensor2lidar_rotation'])
    np.testing.assert_array_equal(s['sensor2lidar_translation'], r['sensor2lidar_translation'])
    assert s['timestamp'] == r['timestamp']
    got = P.load_nuscenes_infos(path, data_root='/data/nusc')
    assert got[0]['lidar_path'] == '/data/nusc/samples/LIDAR_TOP/a.pcd.bin'
    assert got[0]['sweeps'][0]['data_path'] == '/data/nusc/sweeps/LIDAR_TOP/b.pcd.bin'


class _Evil:
    def __reduce__(self):
        return (os.system, ('echo pwned',))


class _Getattr:
    def __reduce__(self):
        return (getattr, ('abc', 'upper'))


@pytest.mark.parametrize('payload', [_Evil(), _Getattr(), pickle.loads])
def test_info_reader_rejects_other_callables(tmp_path, payload):
    path = tmp_path / 'evil.pkl'
    with open(path, 'wb') as f:
        pickle.dump(dict(infos=[dict(lidar_path='a', timestamp=0, sweeps=[], x=payload)]), f)
    with pytest.raises(pickle.UnpicklingError, match='refusing'):
        P.load_nuscenes_infos(str(path))


# ------------------------------------------------------------------------------------- loader host side
def test_loader_capacity_overflow(golden_dir):
    """A file larger than max_points raises before anything reaches a device: nothing is cut silently."""
    loader = P.MultiSweepLoader.from_config(_pipeline_cfg(golden_dir, 'nusc_L'), batch_size=1, max_points=600,
                                            device='cpu')
    rng = np.random.default_rng(5)
    ok = O.make_sample(rng, 500, [580], edges=False)
    loader.read([ok])
    with pytest.raises(ValueError, match='max_points=600'):
        loader.stage([O.make_sample(rng, 601, [10], edges=False)])
    with pytest.raises(ValueError, match='max_points=600'):
        loader.stage([O.make_sample(rng, 10, [100, 601], edges=False)])
    with pytest.raises(ValueError, match='expected 1 samples'):
        loader.read([ok, ok])
    assert loader._dev is None


def test_loader_host_values(golden_dir):
    """Per-source counts, flags, poses and float32 time lags as the reference computes them."""
    loader = P.MultiSweepLoader.from_config(_pipeline_cfg(golden_dir, 'nusc_L'), batch_size=2, max_points=2000,
                                            device='cpu')
    rng = np.random.default_rng(6)
    a, b = O.make_sample(rng, 1000, [900, 0, 700]), O.make_sample(rng, 800, [])
    files, flags, counts, poses, lags = loader.read([a, b])
    assert counts[0].tolist() == [1000 + len(O.edge_points()), 900 + 2 * len(O.edge_points()), 0, 700] + [0] * 7
    assert counts[1].tolist() == [800 + len(O.edge_points())] * 11
    assert flags[0, 0] == P.L.SWEEP_TIME_LAG and flags[0, 1] == 7 and (flags[1, 1:] == 6).all()
    for s, sw in enumerate(a['sweeps'], 1):
        np.testing.assert_array_equal(poses[0, s, :9], sw['sensor2lidar_rotation'].reshape(9))
        assert lags[0, s] == np.float32(a['timestamp'] / 1e6 - sw['timestamp'] / 1e6) and lags[0, s] > 0
    assert lags[0, 0] == 0 and (lags[1] == 0).all() and [r is None for r in files[1]] == [False] + [True] * 10
