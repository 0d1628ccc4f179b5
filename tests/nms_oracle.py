"""Float64 reference of the BEV NMS in get_bboxes(use_nms=True) (srfdet_head.py:1269-1296), for the NMS tests.

TEST INFRASTRUCTURE ONLY, like oracle/: nothing under srfdet_b200/ imports it.  "[3P]" marks third-party semantics
(mmdet3d 1.0.0rc6, mmcv-full 1.7.0 -- neither installed nor vendored) restated from their published sources.
"""
import math

import numpy as np


def _bev_corners(x, y, dx, dy, yaw):
    """Counter-clockwise corners of the footprint: extent dx along u = (cos yaw, sin yaw), dy along v = (-sin yaw, cos yaw)
    (LiDARInstance3DBoxes.bev as mmcv 1.7's box_iou_rotated sees it -- NOT the -yaw sense of boxes3d_to_corners3d)."""
    c, s = math.cos(yaw), math.sin(yaw)
    hx, hy = abs(dx) / 2, abs(dy) / 2
    ux, uy, vx, vy = c * hx, s * hx, -s * hy, c * hy
    return [(x + ux + vx, y + uy + vy), (x - ux + vx, y - uy + vy), (x - ux - vx, y - uy - vy), (x + ux - vx, y + uy - vy)]


def _convex_clip_area(poly, clip):
    """Area of convex polygon `poly` clipped by the convex CCW polygon `clip` (Sutherland-Hodgman, float64)."""
    for e in range(len(clip)):
        (px, py), (qx, qy) = clip[e], clip[(e + 1) % len(clip)]
        ex, ey = qx - px, qy - py
        out = []
        for i in range(len(poly)):
            (ax, ay), (bx, by) = poly[i], poly[(i + 1) % len(poly)]
            da, db = ex * (ay - py) - ey * (ax - px), ex * (by - py) - ey * (bx - px)
            if da >= 0:
                out.append((ax, ay))
            if (da >= 0) != (db >= 0):
                t = da / (da - db)
                out.append((ax + t * (bx - ax), ay + t * (by - ay)))
        if len(out) < 3:
            return 0.0
        poly = out
    s = sum(poly[i][0] * poly[(i + 1) % len(poly)][1] - poly[(i + 1) % len(poly)][0] * poly[i][1] for i in range(len(poly)))
    return max(s / 2, 0.0)


def box_iou_bev(a, b, rotated=True):
    """[3P] mmcv 1.7 ops/box_iou_rotated (rotated) / 2-D nms IoU with offset 0 (rotated=False: axis-aligned dx x dy, yaw
    ignored), restated: IoU of the BEV footprints of box rows (x, y, dx, dy, yaw at columns 0, 1, 3, 4, 6) in float64,
    exact polygon clipping; 0 when either area is below 1e-14.  -> (m, n)."""
    a, b = np.asarray(a, np.float64).reshape(-1, np.shape(a)[-1]), np.asarray(b, np.float64).reshape(-1, np.shape(b)[-1])
    out = np.zeros((a.shape[0], b.shape[0]))
    area_a, area_b = a[:, 3] * a[:, 4], b[:, 3] * b[:, 4]
    ra, rb = np.hypot(a[:, 3], a[:, 4]) / 2, np.hypot(b[:, 3], b[:, 4]) / 2
    d2 = (a[:, None, 0] - b[None, :, 0]) ** 2 + (a[:, None, 1] - b[None, :, 1]) ** 2
    near = (d2 <= (ra[:, None] + rb[None, :]) ** 2) & (area_a[:, None] >= 1e-14) & (area_b[None, :] >= 1e-14)
    for i, j in zip(*np.nonzero(near)):
        p, q = a[i], b[j]
        if rotated:
            sx, sy = (p[0] + q[0]) / 2, (p[1] + q[1]) / 2     # mid-centre shift, as mmcv
            inter = _convex_clip_area(_bev_corners(p[0] - sx, p[1] - sy, p[3], p[4], p[6]),
                                      _bev_corners(q[0] - sx, q[1] - sy, q[3], q[4], q[6]))
        else:
            w = min(p[0] + abs(p[3]) / 2, q[0] + abs(q[3]) / 2) - max(p[0] - abs(p[3]) / 2, q[0] - abs(q[3]) / 2)
            h = min(p[1] + abs(p[4]) / 2, q[1] + abs(q[4]) / 2) - max(p[1] - abs(p[4]) / 2, q[1] - abs(q[4]) / 2)
            inter = max(w, 0.0) * max(h, 0.0)
        out[i, j] = inter / (area_a[i] + area_b[j] - inter)
    return out


def box3d_multiclass_nms(boxes, scores, score_thr, iou_thr, max_num, rotated=True, post_center_range=None, iou=None):
    """[3P] mmdet3d 1.0.0rc6 core/post_processing/box3d_nms.py:box3d_multiclass_nms with mmcv 1.7 ops/iou3d.py nms_bev /
    nms_normal_bev (ops/nms.py), restated (not vendored), for ONE sample of get_bboxes (srfdet_head.py:1269-1296):
    boxes (k, D), scores (k, n_cls) without a background column.  Per class c: candidates scores[:, c] > score_thr sorted by
    score descending (ties: lower index first), greedy keep of every candidate no earlier kept one overlaps with IoU > iou_thr;
    lists concatenated class by class; above max_num the max_num best scores in score order (ties: earlier class-major
    position first); then the post_center_range filter on columns 0..2 (srfdet_head.py get_bboxes), order preserved.
    -> (index (n,), scores (n,), labels (n,))."""
    boxes, scores = np.asarray(boxes, np.float64), np.asarray(scores)
    if iou is None:
        iou = box_iou_bev(boxes, boxes, rotated)
    over = iou > iou_thr
    np.fill_diagonal(over, False)
    idx, sc, lab = [], [], []
    for c in range(scores.shape[1]):
        cand = np.nonzero(scores[:, c] > scores.dtype.type(score_thr))[0]     # compared in the scores' precision
        order = cand[np.lexsort((cand, -scores[cand, c].astype(np.float64)))]
        removed = np.zeros(len(boxes), bool)
        for i in order:
            if removed[i]:
                continue
            idx.append(i)
            sc.append(scores[i, c])
            lab.append(c)
            removed |= over[i]
    idx, sc, lab = np.asarray(idx, np.int64), np.asarray(sc), np.asarray(lab, np.int64)
    if len(idx) > max_num:
        sel = np.lexsort((np.arange(len(idx)), -sc.astype(np.float64)))[:max_num]
        idx, sc, lab = idx[sel], sc[sel], lab[sel]
    if post_center_range is not None and len(idx):
        r = np.asarray(post_center_range, np.float64)
        ctr = boxes[idx, :3]
        keep = (ctr >= r[:3]).all(1) & (ctr <= r[3:]).all(1)
        idx, sc, lab = idx[keep], sc[keep], lab[keep]
    return idx, sc, lab
