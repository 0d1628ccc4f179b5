"""SRFDet / SRFDetWaymo on CUDA: the detector built from the full `model` configs against the measured pipeline
(RegionFeaturePipeline), the reference's head weights through the detector's checkpoint loading, batched inference
(srf_concat_counted_rows), graph replay, image-neck inputs, the simple_test contract and tools/infer.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from srfdet_b200 import synth
from test_oracle_golden import _head_inputs
from util import cuda, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg_path(golden_dir, name):
    return os.path.join(golden_dir, 'configs', 'model', f'srfdet_{name}.py')


def _pipeline_and_detector(golden_dir, name):
    """Calibrated production-size pipeline (scope 'full', use_nms) and a detector from the full config holding its
    point path, backbone, neck and head weights."""
    from srfdet_b200.pipeline import RegionFeaturePipeline
    from srfdet_b200.plugin import SRFDet
    kind, fusion = name.split('_')[0], name.endswith('LC')
    pipe = RegionFeaturePipeline(kind, fusion=fusion, scope='full', use_nms=True)
    pipe.calibrate(cuda(synth.cloud(kind, 44)))
    det = SRFDet.from_config(_cfg_path(golden_dir, name)).cuda()
    sd = dict(pipe.detector.state_dict())
    for prefix, m in (('pts_backbone.', pipe.backbone), ('pts_neck.', pipe.neck), ('bbox_head.', pipe.head)):
        sd.update({prefix + k: v for k, v in m.state_dict().items()})
    res = det.load_checkpoint(sd)
    assert res.missing_keys == [] and res.unexpected_keys == []
    return pipe, det


@pytest.mark.parametrize('name', ['nusc_LC', 'nusc_L', 'waymo_L', 'kitti_L'])
def test_detector_equals_pipeline(golden_dir, name):
    """Same kernels on the same inputs and weights: the detector's infer reproduces the pipeline's frame bit for bit.
    The dynamic-voxel configs (waymo, kitti) average their voxel features with float atomics (DESIGN.md §5), so two runs
    of the same module already differ in the last bits and the chained stages carry that into near-tied NMS rows: they
    are compared on the decoded outputs, in the fp32 mode within 1e-3 (as the batch test)."""
    pipe, det = _pipeline_and_detector(golden_dir, name)
    pts = cuda(synth.cloud(name.split('_')[0], 43))
    if name in ('waymo_L', 'kitti_L'):
        pipe.precision = 'fp32'
        pipe.run_frame(pts)
        det.bbox_head.use_nms = False
        scores, boxes = det.infer([pts], precision='fp32')
        assert rel_err(scores.cpu().numpy(), pipe.last['scores'].cpu().numpy()) < 1e-3
        assert rel_err(boxes.cpu().numpy(), pipe.last['det_boxes'].cpu().numpy()) < 1e-3
        return
    _, ref = pipe.run_frame(pts)                         # (max_per_img, dim-1 + 2): [box | score | label]
    ref_count = pipe.last['nms_count'].clone()
    boxes, scores, labels, counts = det.infer([pts], img_feats=pipe.img_feats, lidar2img=pipe.lidar2img, precision=pipe.precision)
    assert torch.equal(counts, ref_count) and int(counts[0]) > 0
    assert torch.equal(labels[0].float(), ref[:, -1])
    assert torch.equal(boxes[0], ref[:, :-2])
    assert torch.equal(scores[0], ref[:, -2])


_GOLDEN_HEAD_POINT_PATH = dict(
    pts_voxel_layer=dict(max_num_points=10, voxel_size=[0.075, 0.075, 0.2], max_voxels=(120000, 160000),
                         point_cloud_range=[-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]),
    pts_voxel_encoder=dict(type='HardSimpleVFE', num_features=5),
    pts_middle_encoder=dict(type='SparseEncoderCustom', in_channels=5, sparse_shape=[41, 1472, 1472]))


@pytest.mark.parametrize('tag', ['lidar', 'fusion'])
def test_reference_head_weights_through_detector(golden_dir, tag):
    """The reference SRFDetHead's state dict (srfdet_head.npz) loads through the detector's bbox_head. prefix with every
    bbox_head key matched, and the head then reproduces the reference's chained outputs (test_gpu_head_chain.py bounds)."""
    from srfdet_b200.plugin import SRFDet
    z = np.load(os.path.join(golden_dir, 'srfdet_head.npz'))
    params, pf, imf, cfg = _head_inputs(z, tag)
    use_img, C = tag == 'fusion', cfg['C']
    single = dict(type='SingleSRFDetHead' if use_img else 'SingleSRFDetHeadLiDAR', num_cls_convs=2, num_reg_convs=3, dim_feedforward=32,
                  num_heads=2, dropout=0.1, act_cfg=dict(type='ReLU', inplace=True), dynamic_conv=dict(dynamic_dim=4, dynamic_num=2),
                  pc_range=cfg['pc_range'], voxel_size=cfg['voxel_size'], **(dict(use_fusion=True) if use_img else {}))
    roi = lambda s: dict(type='SingleRoIExtractor', roi_layer=dict(type='RoIAlign', output_size=7, sampling_ratio=2), out_channels=C,
                         featmap_strides=s)
    head = dict(type='SRFDetHead', use_img=use_img, num_classes=10, feat_channels_lidar=C, feat_channels_img=C, hidden_dim=C,
                lidar_feat_lvls=4, img_feat_lvls=4, num_proposals=cfg['n_p'], num_heads=cfg['stages'], deep_supervision=True,
                grid_size=[256, 256, 40], out_size_factor=8, code_weights=[1.0] * 8 + [0.2, 0.2], with_dpg=True, num_dpg_exp=4,
                single_head_lidar=single, roi_extractor_lidar=roi([8, 16, 32, 64]), roi_extractor_img=roi([4, 8, 16, 32]))
    det = SRFDet(**_GOLDEN_HEAD_POINT_PATH, bbox_head=head,
                 test_cfg=dict(pts=dict(use_nms=False, max_per_img=20, post_center_range=[-40.0, -40.0, -10.0, 40.0, 40.0, 10.0])))
    det = det.cuda()
    res = det.load_checkpoint({'state_dict': {'bbox_head.' + k: torch.as_tensor(v) for k, v in params.items()}}, strict=False)
    assert not [k for k in res.missing_keys if k.startswith('bbox_head.')] and res.unexpected_keys == []
    pf = [cuda(f) for f in pf]
    imf = [cuda(f) for f in imf] if imf is not None else None
    logits, boxes = det.bbox_head(imf, pf, [dict(lidar2img=z['lidar2img'][0])], precision='fp32')
    tol = 3e-4 if tag == 'lidar' else 1e-3
    np.testing.assert_allclose(logits.cpu().numpy(), z[f'{tag}.logits'], rtol=0, atol=tol)
    np.testing.assert_allclose(boxes.cpu().numpy(), z[f'{tag}.boxes'], rtol=0, atol=tol)
    res = det.bbox_head.get_bboxes(logits, boxes)
    np.testing.assert_array_equal(res[0][2].cpu().numpy(), z[f'{tag}.det_labels'])
    np.testing.assert_allclose(res[0][0].cpu().numpy(), z[f'{tag}.det_boxes'], rtol=0, atol=tol)
    np.testing.assert_allclose(res[0][1].cpu().numpy(), z[f'{tag}.det_scores'], rtol=0, atol=1e-5)


# ---------------------------------------------------------------------------------------- batches
def _concat_ref(blocks, counts, block_rows, width):
    return torch.cat([blocks[b, :max(0, min(int(c), block_rows)), :width] for b, c in enumerate(counts)], 0)


@pytest.mark.parametrize('counts', [[0, 0, 0], [7, 7, 7], [3, 0, 7, 1], [0, 5], [9, -2, 4]])
def test_concat_counted_rows_vs_torch(counts):
    """srf_concat_counted_rows: empty blocks, full blocks, mixed, counts past the block clamp to it, negative to 0;
    two arrays in one launch, one with a column subset; rows past the total stay untouched."""
    from srfdet_b200 import _lib as L
    bs, block_rows = len(counts), 7
    g = torch.Generator().manual_seed(len(counts))
    a = torch.randint(-1000, 1000, (bs, block_rows, 4), generator=g, dtype=torch.int32).cuda()
    b = torch.randn(bs, block_rows, 6, generator=g).cuda()
    d_counts = torch.tensor(counts, dtype=torch.int32).cuda()
    out_a = torch.full((bs * block_rows, 4), 12345, dtype=torch.int32, device='cuda')
    out_b = torch.full((bs * block_rows, 5), 7.0, device='cuda')
    total = torch.full((1,), -1, dtype=torch.int32, device='cuda')
    arrays = (L.Rows * 2)(L.Rows(a.data_ptr(), out_a.data_ptr(), 4, 4, 4), L.Rows(b.data_ptr(), out_b.data_ptr(), 6, 5, 5))
    L.check(L.load().srf_concat_counted_rows(L.ptr(d_counts), bs, block_rows, arrays, 2, L.ptr(total), L.stream_ptr()), 'concat')
    ref_a, ref_b = _concat_ref(a, counts, block_rows, 4), _concat_ref(b, counts, block_rows, 5)
    m = ref_a.shape[0]
    assert int(total) == m
    assert torch.equal(out_a[:m], ref_a) and torch.equal(out_b[:m], ref_b)
    assert bool((out_a[m:] == 12345).all()) and bool((out_b[m:] == 7.0).all())


def test_batch_hard_voxel_equals_single_frames(golden_dir):
    """nusc L (hard voxels): B = 2 in one call equals the two B = 1 calls bit for bit in the packed voxel lists, the BEV maps
    and the FPN pyramid.  The head's final rows are compared at fp32 within 1e-3: the DynamicConv output projection
    splits its reduction over a number of CTAs chosen from the row count (plugin/head.py:_linear, split-K), so its
    sums associate differently at B = 2, and the five chained stages amplify that rounding (DESIGN.md §5)."""
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    clouds = [cuda(synth.cloud('nusc', 50)), cuda(synth.cloud('nusc', 51, n_points=200000))]
    mean, coors, total = det.voxelize_padded(clouds)
    off = 0
    for i, c in enumerate(clouds):
        o = det.pts_voxel_layer.hard_padded(c, batch_idx=0, want_voxels=False, want_mean=True)
        m = int(o['count'])
        single = o['coors'][:m].clone()
        single[:, 0] = i
        assert torch.equal(coors[off:off + m], single) and torch.equal(mean[off:off + m], o['mean'][:m])
        off += m
    assert int(total) == off
    bev2 = det.extract_point_features(clouds)
    pyr2 = det.extract_pts_feat(clouds)
    for i, c in enumerate(clouds):
        assert torch.equal(bev2[i:i + 1], det.extract_point_features([c]))
        for lvl, f in enumerate(det.extract_pts_feat([c])):
            assert torch.equal(pyr2[lvl][i:i + 1], f), lvl
    det.bbox_head.use_nms = False
    sc2, bx2 = [t.clone() for t in det.infer(clouds, precision='fp32')]
    for i, c in enumerate(clouds):
        sc1, bx1 = det.infer([c], precision='fp32')
        assert rel_err(sc2[i].cpu().numpy(), sc1[0].cpu().numpy()) < 1e-3
        assert rel_err(bx2[i].cpu().numpy(), bx1[0].cpu().numpy()) < 1e-3


def test_batch_dynamic_voxel_within_tolerance(golden_dir):
    """waymo L (dynamic voxels, float-atomic voxel means, DESIGN.md §5): B = 2 agrees with the B = 1 runs within the fp16
    tolerance on the BEV maps; the final rows as in the hard-voxel test."""
    _, det = _pipeline_and_detector(golden_dir, 'waymo_L')
    clouds = [cuda(synth.cloud('waymo', 52)), cuda(synth.cloud('waymo', 53, n_points=120000))]
    bev2 = det.extract_point_features(clouds, precision='fp16')
    for i, c in enumerate(clouds):
        assert rel_err(bev2[i].cpu().numpy(), det.extract_point_features([c], precision='fp16')[0].cpu().numpy()) < 1e-2
    det.bbox_head.use_nms = False
    sc2, bx2 = [t.clone() for t in det.infer(clouds, precision='fp32')]
    for i, c in enumerate(clouds):
        sc1, bx1 = det.infer([c], precision='fp32')
        assert rel_err(sc2[i].cpu().numpy(), sc1[0].cpu().numpy()) < 1e-3
        assert rel_err(bx2[i].cpu().numpy(), bx1[0].cpu().numpy()) < 1e-3


def test_graph_replay_equals_eager(golden_dir):
    """One captured B = 2 infer, replayed on two different pairs of clouds, equals the eager result of each pair."""
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    n = 150000
    pairs = [[cuda(synth.cloud('nusc', s)[:n]) for s in (60, 61)], [cuda(synth.cloud('nusc', s)[:n]) for s in (62, 63)]]
    eager = [[t.clone() for t in det.infer(p)] for p in pairs]
    det.use_graph = True
    for p, ref in zip(pairs, eager):
        got = det.infer(p)
        for a, b in zip(got, ref):
            assert torch.equal(a, b)
    assert len(det._graphs) == 1
    assert not torch.equal(eager[0][0], eager[1][0])


def _image_neck_maps(seed, n_cam=6):
    return [cuda(f) for f in synth.feature_pyramid(seed, 256, (232, 400), 4, lead=(1, n_cam))]


def test_lc_image_neck_inputs(golden_dir):
    """nusc LC fed 256-channel image-neck maps: the head's img_convs reduce them, and the result equals feeding the reduced
    128-channel maps; the graph-captured call (which must record the img_convs, not a memo of them) equals both, and so
    does simple_test with lidar2img from img_metas.  More than one cloud with images is refused."""
    pipe, det = _pipeline_and_detector(golden_dir, 'nusc_LC')
    pts = cuda(synth.cloud('nusc', 43))
    maps = _image_neck_maps(70)
    reduced = [f.clone() for f in det.bbox_head._image_maps(maps, pipe.precision)]
    assert [f.shape[2] for f in reduced] == [128] * 4
    a = [t.clone() for t in det.infer([pts], img_feats=maps, lidar2img=pipe.lidar2img)]
    b = [t.clone() for t in det.infer([pts], img_feats=reduced, lidar2img=pipe.lidar2img)]
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    det.use_graph = True
    for feats in (_image_neck_maps(71), maps):         # replay on other maps first, then on the reference ones
        got = det.infer([pts], img_feats=feats, lidar2img=pipe.lidar2img)
    for x, y in zip(got, a):
        assert torch.equal(x, y)
    res = det.simple_test([pts], [dict(lidar2img=pipe.lidar2img.cpu().numpy())], img_feats=maps)
    n = int(a[3][0])
    assert torch.equal(res[0]['pts_bbox']['boxes_3d'], a[0][0, :n].cpu())
    with pytest.raises(NotImplementedError, match='batch-size-1'):
        det.infer([pts, pts], img_feats=maps, lidar2img=pipe.lidar2img)


class _BoxType:
    """Stand-in for mmdet3d's LiDARInstance3DBoxes: (tensor, box_dim) constructor and .to()."""

    def __init__(self, tensor, box_dim):
        self.tensor, self.box_dim = tensor, box_dim

    def to(self, device):
        return _BoxType(self.tensor.to(device), self.box_dim)


def test_simple_test_contract(golden_dir):
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    clouds = [cuda(synth.cloud('nusc', 80)), cuda(synth.cloud('nusc', 81, n_points=100000))]
    boxes, scores, labels, counts = [t.clone() for t in det.infer(clouds)]
    metas = [dict(box_type_3d=_BoxType), dict(box_type_3d=_BoxType)]
    res = det(return_loss=False, points=[clouds], img_metas=[metas])
    assert isinstance(res, list) and len(res) == 2
    for i, r in enumerate(res):
        assert list(r) == ['pts_bbox'] and sorted(r['pts_bbox']) == ['boxes_3d', 'labels_3d', 'scores_3d']
        bx, sc, lb = r['pts_bbox']['boxes_3d'], r['pts_bbox']['scores_3d'], r['pts_bbox']['labels_3d']
        assert isinstance(bx, _BoxType) and bx.box_dim == 9 and bx.tensor.device.type == 'cpu'
        n = int(counts[i])
        assert 0 < n <= 300 and sc.device.type == 'cpu' and lb.device.type == 'cpu' and lb.dtype == torch.int64
        assert torch.equal(bx.tensor, boxes[i, :n].cpu()) and torch.equal(sc, scores[i, :n].cpu())
        assert torch.equal(lb, labels[i, :n].long().cpu())
    plain = det.simple_test(clouds[:1], [{}])
    assert torch.is_tensor(plain[0]['pts_bbox']['boxes_3d'])


def test_tools_infer_end_to_end(golden_dir, tmp_path):
    """tools/infer.py on two .bin clouds and a saved checkpoint equals an in-process simple_test of the same batch."""
    from srfdet_b200.plugin import SRFDet
    cfg = _cfg_path(golden_dir, 'nusc_L')
    torch.manual_seed(5)
    src = SRFDet.from_config(cfg)
    ckpt = str(tmp_path / 'model.pth')
    torch.save({'state_dict': src.state_dict(), 'meta': {'epoch': 1}}, ckpt)
    files = []
    for s, n in ((90, None), (91, 80000)):
        p = str(tmp_path / f'cloud{s}.bin')
        synth.cloud('nusc', s, n_points=n).astype(np.float32).tofile(p)
        files.append(p)
    out = str(tmp_path / 'res.npz')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'), cfg, ckpt, '--points', *files, '--load-dim', '5',
                        '--use-dim', '0', '1', '2', '3', '4', '--precision', 'fp16', '--out', out],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert len([ln for ln in r.stdout.splitlines() if 'cloud9' in ln]) == 2
    det = SRFDet.from_config(cfg).cuda()
    det.load_checkpoint(ckpt)
    ref = det.simple_test([cuda(np.fromfile(f, dtype=np.float32).reshape(-1, 5)) for f in files], [{}, {}])
    got = np.load(out)
    for i, r in enumerate(ref):
        for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
            np.testing.assert_array_equal(got[f'{i}.{k}'], r['pts_bbox'][k].numpy())
