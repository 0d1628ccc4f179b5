"""srf_iou_bev / srf_nms_bev (csrc/nms_bev.cu) against the float64 oracle, graph capture, SRFDetHead.get_bboxes with
use_nms=True, the mmdet3d-signature drop-in and the frame pipeline's opt-in NMS."""
import math

import numpy as np
import pytest
import torch

import nms_oracle
from util import cuda

pytestmark = pytest.mark.gpu

THR = 0.4


def _scene(seed, k, n_cls, dim=9, clusters=60, spread=1.2):
    """Clustered boxes (suppression happens) with distinct scores; any box whose oracle IoU with another lies within 1e-4
    of THR (rotated or axis-aligned) is re-drawn, so fp32 against float64 cannot flip a decision."""
    rng = np.random.default_rng(seed)
    ctr = rng.uniform(-50, 50, (clusters, 2))

    def draw(n):
        b = np.zeros((n, dim), np.float32)
        b[:, :2] = ctr[rng.integers(0, clusters, n)] + rng.normal(0, spread, (n, 2))
        b[:, 2] = rng.uniform(-2, 0, n)
        b[:, 3] = rng.uniform(3.5, 4.8, n)
        b[:, 4] = rng.uniform(1.6, 2.1, n)
        b[:, 5] = rng.uniform(1.4, 1.8, n)
        b[:, 6] = rng.uniform(-math.pi, math.pi, n)
        if dim > 7:
            b[:, 7:] = rng.normal(0, 1, (n, dim - 7))
        return b
    boxes = draw(k)
    for _ in range(20):
        bad = np.zeros(k, bool)
        for rot in (True, False):
            iou = nms_oracle.box_iou_bev(boxes, boxes, rot)
            bad |= (np.abs(iou - THR) < 1e-4).any(1)
        if not bad.any():
            break
        boxes[bad] = draw(int(bad.sum()))
    assert not bad.any()
    scores = (rng.permutation(k * n_cls).reshape(k, n_cls) / (k * n_cls) * 0.98 + 0.01).astype(np.float32)
    return boxes, scores


def _nms_gpu(boxes, scores, score_thr, rotated, max_num, rng=None):
    from srfdet_b200.plugin.nms import nms_device
    out = nms_device(cuda(boxes), cuda(scores), score_thr, THR, rotated, max_num, rng)
    return [t.cpu().numpy() for t in out]


def _check_sample(out, i, boxes, scores, score_thr, rotated, max_num, rng, iou=None):
    ob, osc, olab, oidx, cnt = out
    idx, sc, lab = nms_oracle.box3d_multiclass_nms(boxes, scores, score_thr, THR, max_num, rotated, rng, iou=iou)
    n = int(cnt[i])
    assert n == len(idx), (n, len(idx))
    np.testing.assert_array_equal(oidx[i, :n], idx)
    np.testing.assert_array_equal(olab[i, :n], lab)
    np.testing.assert_array_equal(osc[i, :n], sc)
    np.testing.assert_array_equal(ob[i, :n], boxes[idx])
    assert (olab[i, n:] == -1).all() and (oidx[i, n:] == -1).all() and (osc[i, n:] == 0).all() and (ob[i, n:] == 0).all()
    return n


def _iou_gpu(a, b, rotated):
    from srfdet_b200 import _lib as L
    ta, tb = cuda(a), cuda(b)
    out = torch.empty((a.shape[0], b.shape[0]), device='cuda')
    L.check(L.load().srf_iou_bev(L.ptr(ta), a.shape[0], a.shape[1], L.ptr(tb), b.shape[0], b.shape[1], int(rotated), L.ptr(out),
                                 L.stream_ptr()), 'srf_iou_bev')
    return out.cpu().numpy()


def _row(x, y, dx, dy, yaw):
    return [x, y, 0.0, dx, dy, 1.5, yaw]


@pytest.mark.parametrize('rotated', [True, False])
def test_iou_bev_vs_oracle(rotated):
    hand = np.float32([_row(0.3, -0.2, 2, 1, 0.3), _row(10, 10, 2, 1, 0.3), _row(0, 0, 2, 2, 0), _row(2, 0, 2, 2, 0),
                       _row(0, 0, 4, 4, 0), _row(0.5, 0.5, 1, 2, 0.2), _row(1, 1, 2, 2, 0), _row(0, 0, 2, 2, math.pi / 2),
                       _row(0, 0, 0, 2, 0), _row(0, 0, 4, 1, math.pi / 4), _row(1.5, 1.5, 4, 1, math.pi / 4),
                       _row(55, -55, 0.3, 0.2, 0.4), _row(55.05, -54.97, 0.25, 0.2, -0.3),
                       _row(-55, 55, 0.3, 0.2, 0.4), _row(-54.95, 55.03, 0.25, 0.2, -0.3)])
    g = _iou_gpu(hand, hand, rotated)
    np.testing.assert_allclose(g, nms_oracle.box_iou_bev(hand, hand, rotated), rtol=0, atol=1e-5)
    if rotated:
        assert g[9, 10] == pytest.approx(0.3069, abs=1e-4)         # rotation sense (test_nms_cpu.py::test_rotation_sense)
    boxes, _ = _scene(3, 900, 1)
    g = _iou_gpu(boxes, boxes, rotated)
    ref = nms_oracle.box_iou_bev(boxes, boxes, rotated)
    np.testing.assert_allclose(g, ref, rtol=0, atol=1e-5)
    assert (ref > THR).sum() > 900                                 # the scene really has overlapping pairs


@pytest.mark.parametrize('n_cls,dim', [(10, 9), (3, 7)])
@pytest.mark.parametrize('rotated', [True, False])
def test_nms_bev_vs_oracle(n_cls, dim, rotated):
    scenes = [_scene(10 + s, 900, n_cls, dim) for s in range(2)]
    boxes = np.stack([b for b, _ in scenes])
    scores = np.stack([s for _, s in scenes])
    rng = [-30.0, -30.0, -10.0, 30.0, 30.0, 10.0]
    ious = [nms_oracle.box_iou_bev(b, b, rotated) for b in boxes]
    seen = set()
    for bs in (1, 2):
        for score_thr, max_num in [(0.0, 300), (0.97, 300), (0.0, 10000)]:
            for r in (None, rng):
                out = _nms_gpu(boxes[:bs], scores[:bs], score_thr, rotated, max_num, r)
                for i in range(bs):
                    _check_sample(out, i, boxes[i], scores[i], score_thr, rotated, max_num, r, iou=ious[i])
                    total = len(nms_oracle.box3d_multiclass_nms(boxes[i], scores[i], score_thr, THR, 10 ** 9, rotated, iou=ious[i])[0])
                    seen.add((total > max_num, r is None))
    assert seen == {(True, True), (False, True), (True, False), (False, False)}
    # no candidates at all: count 0, sentinel rows only
    out = _nms_gpu(boxes, scores, 2.0, rotated, 300)
    for i in range(2):
        assert _check_sample(out, i, boxes[i], scores[i], 2.0, rotated, 300, None, iou=ious[i]) == 0


def test_nms_bev_graph_replay():
    from srfdet_b200.plugin.nms import nms_device
    (b0, s0), (b1, s1) = _scene(20, 900, 10), _scene(21, 900, 10)
    boxes, scores = cuda(b0[None]), cuda(s0[None])
    rng = [-40.0, -40.0, -10.0, 40.0, 40.0, 10.0]
    nms_device(boxes, scores, 0.0, THR, True, 300, rng)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = nms_device(boxes, scores, 0.0, THR, True, 300, rng)
    for b, s in [(b1, s1), (b0, s0)]:
        boxes.copy_(cuda(b[None]))
        scores.copy_(cuda(s[None]))
        graph.replay()
        eager = nms_device(boxes, scores, 0.0, THR, True, 300, rng)
        torch.cuda.synchronize()
        for g, e in zip(static_out, eager):
            assert torch.equal(g, e)
        _check_sample([t.cpu().numpy() for t in static_out], 0, b, s, 0.0, True, 300, rng)


def test_get_bboxes_use_nms_golden(golden_dir):
    from test_gpu_head_chain import _build_head, _z
    z = _z(golden_dir, 'srfdet_head.npz')
    head, pf, imf, cfg = _build_head(z, 'lidar')
    head.use_nms = True
    head.test_cfg.update(use_nms=True, max_per_img=20)
    logits, boxes = head(None, [cuda(f) for f in pf], None, precision='fp32')
    with pytest.raises(ValueError):
        head.get_bboxes(logits, boxes)                             # use_nms without nms_thr
    head.test_cfg['nms_thr'] = THR
    res = head.get_bboxes(logits, boxes)
    sc, dec = head.decode(logits, boxes)
    for i, (bx, s, lab) in enumerate(res):
        idx, rs, rl = nms_oracle.box3d_multiclass_nms(dec[i].cpu().numpy(), sc[i].cpu().numpy(), 0.0, THR, 20, True,
                                                  head.test_cfg['post_center_range'])
        assert len(idx) > 0 and lab.dtype == torch.int64
        np.testing.assert_array_equal(lab.cpu().numpy(), rl)
        np.testing.assert_array_equal(s.cpu().numpy(), rs)
        np.testing.assert_array_equal(bx.cpu().numpy(), dec[i].cpu().numpy()[idx])
    calls = []

    def user_nms(bx, s, cfg):
        calls.append(cfg)
        return bx[:3], s[:3, 0], torch.zeros(3, dtype=torch.long, device=bx.device)
    head.nms_fn = user_nms
    res = head.get_bboxes(logits, boxes)
    assert len(calls) == len(res) and all(len(r[0]) <= 3 for r in res)


def test_box3d_multiclass_nms_dropin():
    from srfdet_b200.plugin import box3d_multiclass_nms, xywhr2xyxyr
    from srfdet_b200.plugin.nms import _xyxyr_rows
    b, s = _scene(30, 900, 10)
    mlvl_bboxes = cuda(b)
    for_nms = xywhr2xyxyr(mlvl_bboxes[:, [0, 1, 3, 4, 6]])
    mlvl_scores = torch.cat([cuda(s), torch.rand(900, 1, device='cuda')], dim=1)     # last column: background
    for rot in (True, False):
        bx, sc, lab = box3d_multiclass_nms(mlvl_bboxes, for_nms, mlvl_scores, 0.05, 300, dict(nms_thr=THR, use_rotate_nms=rot))
        rows = _xyxyr_rows(for_nms).cpu().numpy()
        idx, rs, rl = nms_oracle.box3d_multiclass_nms(rows, s, 0.05, THR, 300, rot)
        assert lab.dtype == torch.int64 and len(idx) == 300
        np.testing.assert_array_equal(lab.cpu().numpy(), rl)
        np.testing.assert_array_equal(sc.cpu().numpy(), rs)
        np.testing.assert_array_equal(bx.cpu().numpy(), b[idx])


def test_pipeline_use_nms_frames():
    from srfdet_b200 import synth
    from srfdet_b200.pipeline import RegionFeaturePipeline
    pipe = RegionFeaturePipeline('nusc', fusion=True, scope='full', use_graph=True, use_nms=True)
    pipe.calibrate(cuda(synth.cloud('nusc', 44, n_points=30000)))
    clouds = [cuda(synth.cloud('nusc', 50 + i, n_points=30000)) for i in range(2)]
    outs = [o.clone() for _, o in pipe.run_frames(clouds)]
    torch.cuda.synchronize()
    cfg = pipe.head.test_cfg

    def check_vs_oracle(out):
        sc, dec = pipe.last['scores'][0].cpu().numpy(), pipe.last['det_boxes'][0].cpu().numpy()
        idx, rs, rl = nms_oracle.box3d_multiclass_nms(dec, sc, 0.0, cfg['nms_thr'], cfg['max_per_img'], True, cfg['post_center_range'])
        out = out.cpu().numpy()
        n = len(idx)
        assert out.shape == (300, dec.shape[1] + 2) and n > 0
        np.testing.assert_array_equal(out[:n, -1], rl)
        np.testing.assert_array_equal(out[:n, -2], rs)
        np.testing.assert_array_equal(out[:n, :-2], dec[idx])
        assert (out[n:, -1] == -1).all() and (out[n:, :-1] == 0).all()
    check_vs_oracle(outs[1])                 # self.last: the graph-owned tensors of the last captured slot
    pipe.use_graph = False
    for cloud, out in zip(clouds, outs):
        _, eager = pipe.run_frame(cloud)
        torch.cuda.synchronize()
        assert torch.equal(eager, out)
        check_vs_oracle(eager)
