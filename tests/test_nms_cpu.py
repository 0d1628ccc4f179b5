"""BEV IoU and multi-class NMS of get_bboxes(use_nms=True): the oracle against independent float64 geometry and hand
scenes, and the host side of the drop-ins (no GPU needed)."""
import math

import numpy as np
import pytest
import torch

import nms_oracle


def _box(x, y, dx, dy, yaw):
    return np.array([x, y, 0.0, dx, dy, 1.5, yaw], np.float64)


def _iou(a, b, rotated=True):
    return nms_oracle.box_iou_bev(a[None], b[None], rotated)[0, 0]


def _halfspaces(b):
    x, y, dx, dy, yaw = b[0], b[1], b[3], b[4], b[6]
    u, v = np.array([math.cos(yaw), math.sin(yaw)]), np.array([-math.sin(yaw), math.cos(yaw)])
    c = np.array([x, y])
    rows = []
    for n, h in ((u, dx / 2), (-u, dx / 2), (v, dy / 2), (-v, dy / 2)):
        rows.append([n[0], n[1], -(n @ c) - h])          # n.p - (n.c + h) <= 0
    return np.array(rows)


def _scipy_iou(a, b):
    from scipy.optimize import linprog
    from scipy.spatial import ConvexHull, HalfspaceIntersection
    hs = np.vstack([_halfspaces(a), _halfspaces(b)])
    norm = np.linalg.norm(hs[:, :2], axis=1)
    # Chebyshev centre: an interior point of the intersection, if it has one
    res = linprog([0, 0, -1], A_ub=np.hstack([hs[:, :2], norm[:, None]]), b_ub=-hs[:, 2], bounds=[(None, None)] * 2 + [(0, None)])
    inter = 0.0
    if res.status == 0 and res.x[2] > 1e-9:
        pts = HalfspaceIntersection(hs, res.x[:2]).intersections
        inter = ConvexHull(pts).volume
    return inter / (a[3] * a[4] + b[3] * b[4] - inter)


def test_oracle_iou_vs_halfspace_intersection():
    rng = np.random.default_rng(7)
    worst = 0.0
    for _ in range(1000):
        a = _box(*rng.uniform(-1, 1, 2), *rng.uniform(0.3, 4, 2), rng.uniform(-math.pi, math.pi))
        b = _box(*rng.uniform(-1, 1, 2), *rng.uniform(0.3, 4, 2), rng.uniform(-math.pi, math.pi))
        worst = max(worst, abs(_iou(a, b) - _scipy_iou(a, b)))
    assert worst < 1e-9, worst


def test_oracle_iou_hand_cases():
    a = _box(0.3, -0.2, 2.0, 1.0, 0.3)
    assert _iou(a, a) == pytest.approx(1.0, abs=1e-12)
    assert _iou(a, _box(10, 10, 2, 1, 0.3)) == 0.0
    assert _iou(_box(0, 0, 2, 2, 0), _box(2, 0, 2, 2, 0)) == pytest.approx(0.0, abs=1e-12)      # edge-touching
    big, small = _box(0, 0, 4, 4, 0), _box(0.5, 0.5, 1, 2, 0.2)
    assert _iou(big, small) == pytest.approx(2.0 / 16.0, abs=1e-12)                               # containment: area ratio
    p, q = _box(0, 0, 2, 2, 0), _box(1, 1, 2, 2, 0)
    assert _iou(p, q) == pytest.approx(1.0 / 7.0, abs=1e-12)                                      # axis-aligned closed form
    assert _iou(p, _box(1, 1, 2, 2, 0.7), rotated=False) == pytest.approx(1.0 / 7.0, abs=1e-12)   # yaw ignored
    assert _iou(_box(0, 0, 2, 2, 0), _box(0, 0, 2, 2, math.pi / 2)) == pytest.approx(1.0, abs=1e-12)
    assert _iou(_box(0, 0, 0, 2, 0), _box(0, 0, 0, 2, 0)) == 0.0                                  # zero-size box
    assert _iou(_box(0, 0, 2, 2, 0), _box(0, 0, 2, 0, 0), rotated=False) == 0.0
    for sx, sy in [(55.0, -55.0), (-55.0, 55.0)]:                                                 # small boxes far out
        a, b = _box(sx, sy, 0.3, 0.2, 0.4), _box(sx + 0.05, sy + 0.03, 0.25, 0.2, -0.3)
        assert abs(_iou(a, b) - _scipy_iou(a, b)) < 1e-9


def test_rotation_sense():
    """Extent dx along (cos yaw, sin yaw): B sits 1.5 sqrt 2 further along A's long axis.  Under the -yaw convention of
    boxes3d_to_corners3d the offset would be across the boxes and the IoU 0."""
    a, b = _box(0, 0, 4, 1, math.pi / 4), _box(1.5, 1.5, 4, 1, math.pi / 4)
    inter = 4 - 1.5 * math.sqrt(2)
    assert _iou(a, b) == pytest.approx(inter / (8 - inter), abs=1e-12)
    assert inter / (8 - inter) == pytest.approx(0.3069, abs=1e-4)
    a_neg, b_neg = _box(0, 0, 4, 1, -math.pi / 4), _box(1.5, 1.5, 4, 1, -math.pi / 4)
    assert _iou(a_neg, b_neg) == 0.0


def _nms(boxes, scores, **kw):
    args = dict(score_thr=0.0, iou_thr=0.4, max_num=100, rotated=True)
    args.update(kw)
    return nms_oracle.box3d_multiclass_nms(np.asarray(boxes), np.asarray(scores, np.float32), **args)


def test_oracle_nms_chain():
    """IoU(A, B) = 0.43 and IoU(B, C) = 0.43 > 0.4, IoU(A, C) = 0.11: B is suppressed by A, so C survives."""
    boxes = [_box(0, 0, 2, 1, 0), _box(0.8, 0, 2, 1, 0), _box(1.6, 0, 2, 1, 0)]
    idx, sc, lab = _nms(boxes, [[0.9], [0.8], [0.7]])
    assert idx.tolist() == [0, 2] and lab.tolist() == [0, 0]
    idx, _, _ = _nms(boxes, [[0.7], [0.9], [0.8]])                # B first: it suppresses both neighbours
    assert idx.tolist() == [1]


def test_oracle_nms_score_thr_and_classes():
    boxes = [_box(0, 0, 2, 1, 0), _box(5, 0, 2, 1, 0), _box(10, 0, 2, 1, 0)]
    scores = [[0.5, 0.2], [0.3, 0.6], [0.1, 0.05]]
    idx, sc, lab = _nms(boxes, scores, score_thr=0.1)             # strict: 0.1 is not a candidate
    assert list(zip(idx.tolist(), lab.tolist())) == [(0, 0), (1, 0), (1, 1), (0, 1)]
    np.testing.assert_allclose(sc, np.float32([0.5, 0.3, 0.6, 0.2]))


def test_oracle_nms_max_num():
    boxes = [_box(0, 0, 2, 1, 0), _box(5, 0, 2, 1, 0)]
    scores = [[0.5, 0.1], [0.3, 0.9]]
    idx, sc, lab = _nms(boxes, scores, score_thr=0.2, max_num=3)  # total 3 <= max_num: class-major order
    assert list(zip(idx.tolist(), lab.tolist())) == [(0, 0), (1, 0), (1, 1)]
    idx, sc, lab = _nms(boxes, scores, score_thr=0.2, max_num=2)  # above max_num: best scores, score order
    assert list(zip(idx.tolist(), lab.tolist())) == [(1, 1), (0, 0)]


def test_oracle_nms_equal_scores_and_range():
    boxes = [_box(0, 0, 2, 1, 0), _box(0.1, 0, 2, 1, 0), _box(5, 0, 2, 1, 0)]
    idx, _, _ = _nms(boxes, [[0.5], [0.5], [0.5]])                # equal scores: lower index first, and it suppresses
    assert idx.tolist() == [0, 2]
    idx, _, lab = _nms([_box(0, 0, 2, 1, 0), _box(5, 0, 2, 1, 0)], [[0.7, 0.0], [0.0, 0.7]], max_num=1)
    assert idx.tolist() == [0] and lab.tolist() == [0]           # tie across classes at the cut: earlier class first
    idx, _, _ = _nms(boxes, [[0.5], [0.4], [0.6]], post_center_range=[-1, -1, -1, 1, 1, 1])
    assert idx.tolist() == [0]


def test_dropin_host_side():
    from srfdet_b200.plugin import box3d_multiclass_nms, xywhr2xyxyr
    from srfdet_b200.plugin.nms import _xyxyr_rows
    xywhr = torch.tensor([[1.0, 2.0, 4.0, 2.0, 0.3], [-3.0, 0.5, 1.0, 3.0, -1.0]])
    xyxyr = xywhr2xyxyr(xywhr)
    torch.testing.assert_close(xyxyr, torch.tensor([[-1.0, 1.0, 3.0, 3.0, 0.3], [-3.5, -1.0, -2.5, 2.0, -1.0]]))
    rows = _xyxyr_rows(xyxyr)                                     # back as mmcv converts: centre, extents, angle
    torch.testing.assert_close(rows[:, [0, 1, 3, 4, 6]], xywhr)
    # the last score column is the background: a single column leaves no class, nothing is kept (no device work)
    bx, sc, lab = box3d_multiclass_nms(torch.zeros(3, 9), xyxyr.new_zeros(3, 5), torch.rand(3, 1), 0.0, 10,
                                       dict(nms_thr=0.4, use_rotate_nms=True))
    assert bx.shape == (0, 9) and sc.shape == (0,) and lab.dtype == torch.int64
    with pytest.raises(NotImplementedError):
        box3d_multiclass_nms(torch.zeros(3, 9), xyxyr.new_zeros(3, 5), torch.rand(3, 2), 0.0, 10, dict(nms_thr=0.4),
                             mlvl_dir_scores=torch.zeros(3))
