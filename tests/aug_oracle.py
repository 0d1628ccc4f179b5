"""Reference of test-time augmentation for the LiDAR configs, for the TTA tests.

TEST INFRASTRUCTURE ONLY, like oracle/: nothing under srfdet_b200/ imports it.  "[3P]" marks third-party semantics
(mmdet3d 1.0.0rc6, mmcv-full 1.7.0 -- neither installed nor vendored) restated from their published sources:
datasets/pipelines/test_time_aug.py (MultiScaleFlipAug3D), datasets/pipelines/transforms_3d.py (RandomFlip3D,
GlobalRotScaleTrans, PointsRangeFilter), core/points/lidar_points.py (LiDARPoints.flip), core/bbox/structures/
lidar_box3d.py (LiDARInstance3DBoxes.flip), core/bbox/transforms.py (bbox3d_mapping_back) and
core/post_processing/merge_augs.py (merge_aug_bboxes_3d).  Arithmetic is float32 where torch does it in float32.
"""
import numpy as np

import nms_oracle


def expand_views(pts_scale_ratio=1, flip=False, pcd_horizontal_flip=False, pcd_vertical_flip=False, sync_2d=True,
                 n_img_scale=1, n_flip_direction=1):
    """[3P] MultiScaleFlipAug3D.__call__ with RandomFlip3D inside: -> [(pcd_scale_factor, horizontal, vertical)] in the
    order of the wrapper's loops: img_scale -> pts_scale_ratio -> flip -> pcd_horizontal_flip -> pcd_vertical_flip ->
    flip_direction.  RandomFlip3D(sync_2d=True) sets horizontal = flip and vertical = False; with sync_2d=False it keeps
    the wrapper's pcd flags."""
    ratios = pts_scale_ratio if isinstance(pts_scale_ratio, list) else [float(pts_scale_ratio)]
    flips = [False, True] if flip else [False]
    hs = [False, True] if flip and pcd_horizontal_flip else [False]
    vs = [False, True] if flip and pcd_vertical_flip else [False]
    views = []
    for _ in range(n_img_scale):
        for s in ratios:
            for f in flips:
                for h in hs:
                    for v in vs:
                        for _ in range(n_flip_direction):
                            views.append((s, f, False) if sync_2d else (s, h, v))
    return views


def augment_points(points, scale, horizontal, vertical, point_cloud_range=None):
    """[3P] GlobalRotScaleTrans (identity rotation and translation, points.scale: xyz *= scale in float32), then
    RandomFlip3D (LiDARPoints.flip: horizontal y = -y, vertical x = -x), then PointsRangeFilter (strict lo < p < hi on
    x, y, z) when a range is given.  points (n, C) float32 -> (n', C) float32."""
    p = np.array(points, np.float32, copy=True)
    p[:, :3] = p[:, :3] * np.float32(scale)
    if horizontal:
        p[:, 1] = -p[:, 1]
    if vertical:
        p[:, 0] = -p[:, 0]
    if point_cloud_range is not None:
        r = np.asarray(point_cloud_range, np.float32)
        keep = ((p[:, :3] > r[:3]) & (p[:, :3] < r[3:])).all(1)
        p = p[keep]
    return p


def bbox3d_mapping_back(boxes, scale, horizontal, vertical):
    """[3P] bbox3d_mapping_back on LiDARInstance3DBoxes rows [x, y, z, dx, dy, dz, yaw (, vx, vy)], float32:
    horizontal: columns 1::7 negated, then yaw = -yaw; vertical: columns 0::7 negated, then yaw = -yaw + pi (np.pi added
    to a float32 tensor: fl32(pi)); then columns [:6] and [7:] times fl32(1 / scale)."""
    b = np.array(boxes, np.float32, copy=True)
    if horizontal:
        b[:, 1::7] = -b[:, 1::7]
        b[:, 6] = -b[:, 6]
    if vertical:
        b[:, 0::7] = -b[:, 0::7]
        b[:, 6] = -b[:, 6] + np.float32(np.pi)
    inv = np.float32(1 / scale)
    b[:, :6] = b[:, :6] * inv
    b[:, 7:] = b[:, 7:] * inv
    return b


def merge_aug_bboxes_3d(results, views, nms_thr, max_num, rotated=True):
    """[3P] merge_aug_bboxes_3d for one sample: results [(boxes (n_a, D) float32, scores (n_a,), labels (n_a,))] per view
    in meta order, views [(scale, horizontal, vertical)].  Every view mapped back and concatenated; per class, greedy NMS
    (nms_bev / nms_normal_bev) in (score desc, concatenated position asc) order, suppression at IoU > nms_thr; kept lists
    concatenated class-major and sorted by score descending (ties: class-major position asc); the first
    min(max_num, total).  -> (boxes, scores, labels, concatenated positions)."""
    boxes = np.concatenate([bbox3d_mapping_back(b, *v) for (b, _, _), v in zip(results, views)]).astype(np.float32)
    scores = np.concatenate([np.asarray(s, np.float32) for _, s, _ in results])
    labels = np.concatenate([np.asarray(lab, np.int64) for _, _, lab in results])
    pos = []
    for c in (range(int(labels.max()) + 1) if len(labels) else []):
        cand = np.nonzero(labels == c)[0]
        if len(cand) == 0:
            continue
        order = cand[np.lexsort((cand, -scores[cand].astype(np.float64)))]
        over = nms_oracle.box_iou_bev(boxes[order], boxes[order], rotated) > nms_thr
        removed = np.zeros(len(order), bool)
        for i in range(len(order)):
            if removed[i]:
                continue
            pos.append(order[i])
            removed[i + 1:] |= over[i, i + 1:]
    pos = np.asarray(pos, np.int64)
    sel = np.lexsort((np.arange(len(pos)), -scores[pos].astype(np.float64)))[:min(max_num, len(pos))]
    pos = pos[sel]
    return boxes[pos], scores[pos], labels[pos], pos


def bev_footprint(box):
    """Corners of a box row's BEV footprint (nms_oracle's rotation sense), float64."""
    b = np.asarray(box, np.float64)
    return np.asarray(nms_oracle._bev_corners(b[0], b[1], b[3], b[4], b[6]))
