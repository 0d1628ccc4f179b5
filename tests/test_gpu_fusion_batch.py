"""Batched camera fusion on CUDA: a batch of B fusion samples is B independent batch-1 calls (SURVEY.md §3.4), each
sample with its own clouds, image maps and lidar2img.  Every batched case rotates each sample's camera rig
(synth.lidar2img(yaw_offsets=)) and draws its own maps and boxes, and checks that the samples' outputs differ, so a
kernel that read sample 0's cameras for every sample fails."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import oracle as O
from srfdet_b200 import synth
from test_gpu_detector import _cfg_path, _pipeline_and_detector
from util import cuda

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PC = [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0]
YAWS = [0.0, 0.45, -0.8, 1.2]
HW = (232, 400)


def _pooler(c, strides=(4, 8, 16, 32)):
    from srfdet_b200.plugin import SingleRoIExtractor
    return SingleRoIExtractor(dict(type='RoIAlign', output_size=7, sampling_ratio=2), c, list(strides))


def _maps(seed, b, n_cam, c, channels_last):
    """(b, n_cam, c, H_l, W_l) N(0,1) maps drawn on the device; channels_last: NHWC images packed densely."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    out, (h, w) = [], HW
    for _ in range(4):
        f = torch.randn((b * n_cam, c, h, w), generator=g, device='cuda')
        if channels_last:
            f = f.contiguous(memory_format=torch.channels_last)
        out.append(f.view(b, n_cam, c, h, w))
        h, w = (h + 1) // 2, (w + 1) // 2
    return out


def _l2i(b, n_cam=6):
    return cuda(synth.lidar2img(n_cam, b, yaw_offsets=YAWS[:b]))


def _chained_rows_agree(got, ref, tol=1e-3, max_frac=0.1):
    """Decoded rows of the five chained stages: B > 1 against B = 1.  The first stage's features are bit-identical (tested
    below); later stages differ in the last bits because the DynamicConv output projection picks its split-K from the row
    count (plugin/head.py:_linear).  The camera branch turns such last-bit changes into jumps for a few proposals (a
    projected rectangle that crosses a FPN level or image-border threshold samples other pixels in the next stage), so the
    bound is per proposal: most rows within tol of max |ref|, and a tiny median.  Measured on a B200 for these inputs:
    at most 5.3 % of rows above 1e-3 (B = 4), medians up to 1.6e-5, the worst row 8.8e-2.  Reading another sample's
    cameras moves every row by O(1), far past the median bound."""
    g = got.cpu().numpy().reshape(got.shape[0], -1).astype(np.float64)
    r = ref.cpu().numpy().reshape(ref.shape[0], -1).astype(np.float64)
    err = np.abs(g - r).max(1) / max(np.abs(r).max(), 1e-12)
    assert (err > tol).mean() <= max_frac and np.median(err) < 1e-4, ((err > tol).mean(), float(np.median(err)), float(err.max()))


def _bits(t):
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)


# ---------------------------------------------------------------------------------------- kernel
FORMS = [('nchw', 'f32'), ('nchw', 'f32_nchw_out'), ('cl', 'f32'), ('cl', 'f32_off'), ('cl', 'f16_off'), ('cl', 'f16x2_off')]


@pytest.mark.parametrize('form', FORMS, ids=['-'.join(f) for f in FORMS])
@pytest.mark.parametrize('c', [128, 256])
@pytest.mark.parametrize('n_cam', [1, 6])
@pytest.mark.parametrize('batch', [1, 2, 3])
def test_img_roi_batch_equals_single_calls(batch, n_cam, c, form):
    """srf_img_roi_features over B samples equals B batch-1 calls bit for bit: the features (every output form, at a channel
    offset into a wider row for the *_off forms) and the image RoIs, whose column 0 moves by b * n_cam."""
    from srfdet_b200 import _lib as L
    from srfdet_b200.plugin import img_feats_sampling_bboxes_roi
    layout, out_form = form
    n_p = 300
    maps = _maps(10 * batch + n_cam + c, batch, n_cam, c, layout == 'cl')
    boxes = cuda(synth.proposals(40 + batch, n_p, 10, batch))
    l2i = _l2i(batch, n_cam)
    pool = _pooler(c)
    enc = {'f16_off': L.F16, 'f16x2_off': L.F16X2}.get(out_form, L.F32)
    off = 8 if out_form.endswith('_off') else 0

    def run(m, b, p, k):
        kw = dict(channel_last=out_form != 'f32_nchw_out', return_rois=True)
        if off:
            buf = torch.full((k, 49, L.enc_width(enc, c + 2 * off)), 7.0, dtype=L.enc_torch_dtype(enc), device='cuda')
            kw.update(out=buf, ch_offset=off, out_enc=enc)
        return img_feats_sampling_bboxes_roi(m, b, pool, p, PC, **kw)
    got, rois = run(maps, boxes, l2i, batch * n_p)
    for b in range(batch):
        one, one_rois = run([f[b:b + 1] for f in maps], boxes[b:b + 1], l2i[b], n_p)
        assert torch.equal(_bits(got[b * n_p:(b + 1) * n_p]), _bits(one)), b
        mine = rois.view(batch, n_cam * n_p, 5)[b].clone()
        assert torch.equal(mine[:, 1:], one_rois[:, 1:]), b
        assert torch.equal(mine[:, 0], one_rois[:, 0] + b * n_cam), b
    assert torch.equal(boxes, cuda(synth.proposals(40 + batch, n_p, 10, batch)))       # not mutated
    if batch > 1:
        assert not torch.equal(got[:n_p], got[n_p:2 * n_p])
        assert float(got[n_p:2 * n_p].float().abs().sum()) > 0


def test_img_roi_batch_non_dense_maps():
    """Levels whose images are not densely packed (a crop of wider maps) are copied, never read with strides the kernel
    does not assume: the result equals the densely packed maps'."""
    from srfdet_b200.plugin import img_feats_sampling_bboxes_roi
    wide = _maps(5, 2, 6, 128, True)
    crop = [f[..., :f.shape[-1] - 3] for f in wide]
    dense = [f.clone(memory_format=torch.contiguous_format) for f in crop]
    boxes, l2i = cuda(synth.proposals(6, 200, 10, 2)), _l2i(2)
    for cl in (False, True):
        a = img_feats_sampling_bboxes_roi(crop, boxes, _pooler(128), l2i, PC, channel_last=cl)
        b = img_feats_sampling_bboxes_roi(dense, boxes, _pooler(128), l2i, PC, channel_last=cl)
        assert torch.equal(a, b)


def test_img_roi_batch_vs_oracle_per_sample():
    """The fp32 output of each sample of a B = 2 call matches the oracle run on that sample alone at B = 1, within the
    bounds of test_gpu_roi_head.py::test_img_roi_production_size_vs_oracle.  (The oracle is not called with B > 1: it
    reproduces the reference's inconsistent batch indexing.)"""
    from srfdet_b200.plugin import img_feats_sampling_bboxes_roi
    C, B, n_p = 32, 2, 900
    feats = [synth.hash_field((B, 6, C, 232 // 2 ** i, 400 // 2 ** i), 70 + i) for i in range(4)]
    boxes = synth.proposals(9, n_p, 10, B)
    l2i = synth.lidar2img(6, B, yaw_offsets=YAWS[:B])
    got, rois = img_feats_sampling_bboxes_roi([cuda(f) for f in feats], cuda(boxes), _pooler(C), cuda(l2i), PC, return_rois=True)
    got, rois = got.cpu().numpy(), rois.cpu().numpy().reshape(B, 6 * n_p, 5)
    assert np.abs(got[:n_p] - got[n_p:]).max() > 0
    for b in range(B):
        ref = O.img_roi_feats([f[b:b + 1] for f in feats], boxes[b:b + 1], l2i[b:b + 1], PC, [4, 8, 16, 32])
        ref_rois = O.img_rois(boxes[b:b + 1], l2i[b:b + 1], PC).numpy()
        np.testing.assert_array_equal(rois[b][:, 0], ref_rois[:, 0] + b * 6)
        r_got, r_ref = rois[b][:, 1:], ref_rois[:, 1:]
        near = np.abs(r_ref) < 2e3
        np.testing.assert_allclose(r_got[near], r_ref[near], rtol=2e-4, atol=2e-2)
        np.testing.assert_allclose(r_got[~near], r_ref[~near], rtol=2e-2)
        err = np.abs(got[b * n_p:(b + 1) * n_p] - ref).reshape(n_p, -1).max(1)
        assert (err > 2e-3).sum() <= 4, (b, (err > 2e-3).sum())
        assert np.median(err) < 1e-4
        assert (np.abs(ref).reshape(n_p, -1).max(1) > 0).sum() > 300


# ---------------------------------------------------------------------------------------- head and detector
@pytest.fixture(scope='module')
def lc(golden_dir):
    pipe, det = _pipeline_and_detector(golden_dir, 'nusc_LC')
    det.bbox_head.use_nms = False
    clouds = [cuda(synth.cloud('nusc', 200 + i)) for i in range(4)]
    return pipe, det, clouds


def test_head_batch_equals_single(lc):
    """SRFDetHead at B = 2: the image half of DPG and the first stage's fused RoI features equal the B = 1 runs bit for bit;
    the decoded rows after the five stages agree within 1e-3 in fp32 (the DynamicConv output projection's split-K sums
    associate differently at another row count, see test_batch_hard_voxel_equals_single_frames); the camera branch makes
    a few proposals jump on such last-bit changes, so the bound is per proposal (_chained_rows_agree)."""
    _, det, clouds = lc
    head = det.bbox_head
    maps, l2i = _maps(300, 2, 6, 128, True), _l2i(2)
    pyr = det.extract_pts_feat(clouds[:2], 'fp32')
    dpg2 = head.dpg_image_logits(maps)
    dpg1 = [head.dpg_image_logits([f[b:b + 1] for f in maps]) for b in range(2)]
    for b in range(2):
        assert torch.equal(dpg2[b:b + 1], dpg1[b])
    assert not torch.equal(dpg2[0], dpg2[1])
    boxes, _ = head._get_init_proposals(maps, pyr, sigmoid_centres=True)
    stage = head.head_series_lidar[0]

    def roi(m, p, bx, l):
        return stage.region_features(m, p, bx.clone(), head.roi_extractor_lidar, head.roi_extractor_img, l, 'fp32')
    r2 = roi(maps, pyr, boxes, l2i)
    n_p = boxes.shape[1]
    for b in range(2):
        r1 = roi([f[b:b + 1] for f in maps], [p[b:b + 1] for p in pyr], boxes[b:b + 1], l2i[b])
        assert torch.equal(r2[b * n_p:(b + 1) * n_p], r1), b
    assert not torch.equal(r2[:n_p], r2[n_p:])
    sc2, bx2 = head.decode(*head(maps, pyr, None, lidar2img=l2i, precision='fp32'))
    for b in range(2):
        one = [p[b:b + 1] for p in pyr]
        sc1, bx1 = head.decode(*head([f[b:b + 1] for f in maps], one, None, lidar2img=l2i[b], precision='fp32'))
        _chained_rows_agree(sc2[b], sc1[0])
        _chained_rows_agree(bx2[b], bx1[0])


@pytest.mark.parametrize('batch', [2, 4])
def test_detector_batch_equals_single(lc, batch):
    """nusc LC infer at B = 2 and 4 (use_nms=False, fp32): the FPN pyramid of each sample is bit-identical to its B = 1
    run, the scores and boxes agree per proposal as in test_head_batch_equals_single, and 256-channel image-neck maps through img_convs equal the reduced
    128-channel maps."""
    _, det, all_clouds = lc
    clouds = all_clouds[:batch]
    pyr = det.extract_pts_feat(clouds, 'fp32')
    for b, c in enumerate(clouds):
        for lvl, f in enumerate(det.extract_pts_feat([c], 'fp32')):
            assert torch.equal(pyr[lvl][b:b + 1], f), (b, lvl)
    maps, l2i = _maps(400 + batch, batch, 6, 128, True), _l2i(batch)
    sc, bx = [t.clone() for t in det.infer(clouds, img_feats=maps, lidar2img=l2i, precision='fp32')]
    for b, c in enumerate(clouds):
        sc1, bx1 = det.infer([c], img_feats=[f[b:b + 1] for f in maps], lidar2img=l2i[b], precision='fp32')
        _chained_rows_agree(sc[b], sc1[0])
        _chained_rows_agree(bx[b], bx1[0])
    assert not torch.equal(sc[0], sc[1])
    wide = _maps(500 + batch, batch, 6, 256, False)
    reduced = [f.clone() for f in det.bbox_head._image_maps(wide, 'fp32')]
    assert [f.shape[2] for f in reduced] == [128] * 4
    a = [t.clone() for t in det.infer(clouds, img_feats=wide, lidar2img=l2i, precision='fp32')]
    b = det.infer(clouds, img_feats=reduced, lidar2img=l2i, precision='fp32')
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_graph_replay_batched_fusion(lc):
    """One captured B = 2 infer, replayed on two different (clouds, maps, lidar2img) sets, equals the eager result of each."""
    _, det, clouds = lc
    sets = [(clouds[:2], _maps(600, 2, 6, 128, True), _l2i(2)),
            (clouds[2:4], _maps(601, 2, 6, 128, True), cuda(synth.lidar2img(6, 2, yaw_offsets=[0.9, -0.3])))]
    det.reset_graphs()
    eager = [[t.clone() for t in det.infer(p, img_feats=m, lidar2img=l)] for p, m, l in sets]
    det.use_graph = True
    try:
        for (p, m, l), ref in zip(sets, eager):
            got = det.infer(p, img_feats=m, lidar2img=l)
            for x, y in zip(got, ref):
                assert torch.equal(x, y)
        assert len(det._graphs) == 1
    finally:
        det.use_graph = False
        det.reset_graphs()
    assert not torch.equal(eager[0][0], eager[1][0])


def _swap(maps):
    out = []
    for f in maps:
        s = torch.empty_like(f)
        s[0], s[1] = f[1], f[0]
        out.append(s)
    return out


def test_simple_test_takes_each_samples_lidar2img(lc):
    """simple_test / forward_test at B = 2 read each sample's lidar2img from its own meta and equal the infer rows;
    swapping the metas together with the clouds and the map slices swaps the results."""
    _, det, clouds = lc
    det.bbox_head.use_nms = True
    try:
        pts, maps, l2i = clouds[:2], _maps(700, 2, 6, 128, True), _l2i(2)
        boxes, scores, labels, counts = [t.clone() for t in det.infer(pts, img_feats=maps, lidar2img=l2i)]
        metas = [dict(lidar2img=l2i[b].cpu().numpy()) for b in range(2)]
        res = det.simple_test(pts, metas, img_feats=maps)
        same = det(return_loss=False, points=[pts], img_metas=[metas], img_feats=maps)
        for b in range(2):
            n = int(counts[b])
            assert n > 0
            r = res[b]['pts_bbox']
            assert torch.equal(r['boxes_3d'], boxes[b, :n].cpu()) and torch.equal(r['scores_3d'], scores[b, :n].cpu())
            assert torch.equal(r['labels_3d'], labels[b, :n].long().cpu())
            for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
                assert torch.equal(same[b]['pts_bbox'][k], r[k])
        assert not torch.equal(res[0]['pts_bbox']['scores_3d'][:5], res[1]['pts_bbox']['scores_3d'][:5])
        swapped = det.simple_test(pts[::-1], metas[::-1], img_feats=_swap(maps))
        for b in range(2):
            for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
                assert torch.equal(swapped[1 - b]['pts_bbox'][k], res[b]['pts_bbox'][k]), (b, k)
        # the same clouds and maps with only the metas swapped: the projections follow the metas
        crossed = det.simple_test(pts, metas[::-1], img_feats=maps)
        assert not torch.equal(crossed[0]['pts_bbox']['scores_3d'], res[0]['pts_bbox']['scores_3d'])
    finally:
        det.bbox_head.use_nms = False


def test_tools_infer_batched_fusion(golden_dir, tmp_path):
    """tools/infer.py with two .bin clouds, a (2, 6, C, H, W) .npz of image maps and a (2, 6, 4, 4) .npy equals the
    in-process simple_test of the same batch."""
    from srfdet_b200.plugin import SRFDet, registry, set_precision
    cfg = _cfg_path(golden_dir, 'nusc_LC')
    torch.manual_seed(6)
    src = SRFDet.from_config(cfg)
    ckpt = str(tmp_path / 'model.pth')
    torch.save({'state_dict': src.state_dict()}, ckpt)
    files = []
    for s, n in ((92, None), (93, 90000)):
        p = str(tmp_path / f'cloud{s}.bin')
        synth.cloud('nusc', s, n_points=n).astype(np.float32).tofile(p)
        files.append(p)
    maps = synth.feature_pyramid(94, 128, HW, 4, lead=(2, 6))
    l2i = synth.lidar2img(6, 2, yaw_offsets=YAWS[:2])
    np.savez(str(tmp_path / 'maps.npz'), **{f'level{i}': f for i, f in enumerate(maps)})
    np.save(str(tmp_path / 'l2i.npy'), l2i)
    out = str(tmp_path / 'res.npz')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'), cfg, ckpt, '--points', *files,
                        '--img-feats', str(tmp_path / 'maps.npz'), '--lidar2img', str(tmp_path / 'l2i.npy'),
                        '--precision', 'fp16', '--out', out], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    det = SRFDet.from_config(cfg).cuda()
    det.load_checkpoint(ckpt)
    old = registry.get_precision()
    set_precision('fp16')
    try:
        ref = det.simple_test([cuda(np.fromfile(f, dtype=np.float32).reshape(-1, 5)) for f in files],
                              [dict(lidar2img=l2i[b]) for b in range(2)], img_feats=[cuda(f) for f in maps])
    finally:
        set_precision(old)
    got = np.load(out)
    for i, r in enumerate(ref):
        for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
            np.testing.assert_array_equal(got[f'{i}.{k}'], r['pts_bbox'][k].numpy())
