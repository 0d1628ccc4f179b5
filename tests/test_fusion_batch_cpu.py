"""Batched camera fusion, host side (no GPU needed): the detector's and the sampler's argument checks run before any
device work, tools/infer.py's camera inputs, the C entry point's batch check and the profiler's work model of
srf_img_roi_features."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def det(golden_dir):
    from srfdet_b200.plugin import SRFDet, load_config
    return SRFDet.from_config(load_config(os.path.join(golden_dir, 'configs', 'model', 'srfdet_nusc_LC.py'))['model'])


def _maps(b, n_cam=6, c=128, levels=4):
    return [torch.zeros(b, n_cam, c, 8 >> i, 8 >> i) for i in range(levels)]


def _l2i(*lead):
    return torch.eye(4).expand(*lead, 4, 4).clone()


def test_one_camera_set_for_several_clouds_is_refused(det):
    """Two clouds with maps of batch 1 and one (n_cam, 4, 4) set: the reference's undefined B > 1 case."""
    pts = [torch.zeros(4, 5)] * 2
    for l2i in (_l2i(6), _l2i(1, 6)):
        with pytest.raises(NotImplementedError, match='batch-size-1') as e:
            det.infer(pts, img_feats=_maps(1), lidar2img=l2i)
        assert '(2, 6, 4, 4)' in str(e.value) and '(2, 6, C, H, W)' in str(e.value)


@pytest.mark.parametrize('case', ['maps_batch', 'maps_batch_one_set', 'levels_disagree', 'l2i_batch', 'l2i_one_set',
                                  'l2i_cams', 'maps_4d', 'too_many'])
def test_fusion_batch_argument_checks(det, case):
    n = 9 if case == 'too_many' else 2
    pts = [torch.zeros(4, 5)] * n
    maps, l2i = _maps(n), _l2i(n, 6)
    match = None
    if case == 'maps_batch':
        maps, match = _maps(3), 'batch 3 for 2 clouds'
    elif case == 'maps_batch_one_set':          # maps of batch 1 but two camera sets: the batches disagree
        maps, match = _maps(1), 'batch 1 for 2 clouds'
    elif case == 'levels_disagree':
        maps, match = _maps(2)[:3] + _maps(3)[3:], 'same batch'
    elif case == 'l2i_batch':
        l2i, match = _l2i(3, 6), r'\(2, 6, 4, 4\)'
    elif case == 'l2i_one_set':
        l2i, match = _l2i(6), r'\(2, 6, 4, 4\)'
    elif case == 'l2i_cams':
        l2i, match = _l2i(2, 5), r'\(2, 6, 4, 4\)'
    elif case == 'maps_4d':
        maps, match = [f[0] for f in maps], 'B, n_cam, C, H, W'
    elif case == 'too_many':
        match = 'at most 8 samples'
    with pytest.raises(ValueError, match=match):
        det.infer(pts, img_feats=maps, lidar2img=l2i)


def test_simple_test_needs_a_meta_per_sample(det):
    pts = [torch.zeros(4, 5)] * 2
    with pytest.raises(ValueError, match='its own meta'):
        det.simple_test(pts, [dict(lidar2img=np.eye(4, dtype=np.float32)[None].repeat(6, 0))], img_feats=_maps(2))


def test_fusion_tta_still_refused(det):
    metas = [dict(lidar2img=np.eye(4, dtype=np.float32)[None].repeat(6, 0))] * 2
    with pytest.raises(NotImplementedError, match='augmentation'):
        det.forward_test(points=[[torch.zeros(4, 5)] * 2] * 2, img_metas=[metas, metas], img_feats=_maps(2))


def test_sampler_shape_checks():
    """img_feats_sampling_bboxes_roi rejects mismatched batches and projections before touching the device."""
    from srfdet_b200.plugin import SingleRoIExtractor, img_feats_sampling_bboxes_roi
    pool = SingleRoIExtractor(dict(type='RoIAlign', output_size=7, sampling_ratio=2), 128, [4, 8, 16, 32])
    pc = [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]
    boxes = torch.zeros(2, 10, 10)
    with pytest.raises(ValueError, match='for 2 samples'):
        img_feats_sampling_bboxes_roi(_maps(3), boxes, pool, _l2i(2, 6), pc)
    with pytest.raises(ValueError, match=r'pass \(2, 6, 4, 4\)'):
        img_feats_sampling_bboxes_roi(_maps(2), boxes, pool, _l2i(6), pc)
    with pytest.raises(ValueError, match=r'pass \(2, 6, 4, 4\)'):
        img_feats_sampling_bboxes_roi(_maps(2), boxes, pool, _l2i(2, 4), pc)
    with pytest.raises(ValueError, match='same number of cameras'):
        img_feats_sampling_bboxes_roi(_maps(2)[:2] + _maps(2, n_cam=5)[2:], boxes, pool, _l2i(2, 6), pc)
    with pytest.raises(ValueError, match='B, n_cam, C, H, W'):
        img_feats_sampling_bboxes_roi([f[0] for f in _maps(2)], boxes, pool, _l2i(2, 6), pc)


def test_flat_image_maps_are_views():
    """The img_convs output layout (NHWC rows viewed as (B, n_cam, C, H, W)) and NCHW maps flatten to
    (B*n_cam, C, H, W) without a copy; the channels_last test holds for the flattened maps."""
    from srfdet_b200.plugin.roi import flat_image_maps, maps_channels_last
    rows = torch.randn(2 * 6 * 5 * 7, 16)
    cl = rows.view(2, 6, 5, 7, 16).permute(0, 1, 4, 2, 3)
    nchw = torch.randn(2, 6, 16, 5, 7)
    for f in (cl, nchw):
        flat = flat_image_maps([f])[0]
        assert flat.shape == (12, 16, 5, 7) and flat.data_ptr() == f.data_ptr()
        assert torch.equal(flat[7], f[1, 1])
    assert maps_channels_last(flat_image_maps([cl])) and not maps_channels_last(flat_image_maps([nchw]))
    crop = cl[..., :6]
    assert not maps_channels_last(flat_image_maps([crop]))


def _infer_tool():
    spec = importlib.util.spec_from_file_location('srfdet_infer_tool', os.path.join(ROOT, 'tools', 'infer.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_tools_infer_camera_inputs():
    tool = _infer_tool()
    z4 = {f'l{i}': np.zeros((6, 8, 4 >> i, 4 >> i), np.float32) for i in range(3)}
    z5 = {k: np.stack([v, v]) for k, v in z4.items()}

    class Npz(dict):
        @property
        def files(self):
            return list(self)
    maps, l2i = tool.camera_inputs(Npz(z4), np.eye(4)[None].repeat(6, 0), 1)
    assert [m.shape[:2] for m in maps] == [(1, 6)] * 3 and l2i.shape == (1, 6, 4, 4)
    maps, l2i = tool.camera_inputs(Npz(z5), np.eye(4)[None, None].repeat(2, 0).repeat(6, 1), 2)
    assert [m.shape[:2] for m in maps] == [(2, 6)] * 3 and l2i.shape == (2, 6, 4, 4)
    for z, l2i, n, msg in [(z4, np.eye(4)[None].repeat(6, 0), 2, 'sample'),             # one sample of maps for 2 clouds
                           (z5, np.eye(4)[None].repeat(6, 0), 2, 'lidar2img'),          # one camera set for 2 clouds
                           (z5, np.eye(4)[None, None].repeat(2, 0).repeat(5, 1), 2, 'lidar2img'),
                           (z5, np.eye(4)[None, None].repeat(2, 0).repeat(6, 1), 3, 'sample')]:
        with pytest.raises(SystemExit, match=msg):
            tool.camera_inputs(Npz(z), l2i, n)


def test_img_roi_entry_point_rejects_batch_below_one():
    """srf_img_roi_features: batch < 1 is SRF_ERR_ARG with a message, returned before any launch."""
    from srfdet_b200 import _lib as L
    from srfdet_b200 import build
    build.build()
    lib = L.load()
    p = L.Pyramid()
    p.n_levels, p.channels, p.channels_last = 1, 128, 0
    p.feat[0], p.h[0], p.w[0], p.stride[0] = 256, 8, 8, 4.0          # never dereferenced
    out = L.RoiOut(256, 1, L.F32, 128, 0)
    for batch in (0, -1):
        rc = lib.srf_img_roi_features(ctypes.byref(p), 256, batch, 10, 10, 256, 6, L.f6([0] * 6), ctypes.byref(out), None, None)
        assert rc == -1 and b'batch' in lib.srf_last_error()


def test_profiler_work_of_img_roi_features():
    """bench.py's kernel table: the image RoIAlign bytes of a batch-1 call are those of the parent's work model, and a batch
    of B counts B samples."""
    from srfdet_b200 import _lib as L
    from srfdet_b200.profiling import _work
    s = dict(channels=128, hw=[(232, 400), (116, 200), (58, 100), (29, 50)], out_enc=L.BF16X2)
    ctx = dict(n_points=1, c_points=5, img_roi_input_bytes=63_000_000)
    a1 = (None, None, 1, 900, 10, None, 6, None, None, None, None)
    assert _work('srf_img_roi_features', a1, s, ctx) == (0.0, 900 * 49 * 128 * 4 + 63_000_000)
    a4 = (None, None, 4, 900, 10, None, 6, None, None, None, None)
    assert _work('srf_img_roi_features', a4, s, ctx) == (0.0, 4 * (900 * 49 * 128 * 4 + 63_000_000))
    full = 6 * sum(h * w for h, w in s['hw']) * 128 * 4
    assert _work('srf_img_roi_features', a1, s, dict(n_points=1, c_points=5)) == (0.0, 900 * 49 * 128 * 4 + full)
