"""BEV NMS drop-ins under the names the reference imports (mmdet3d.core: xywhr2xyxyr, box3d_multiclass_nms;
mmcv.ops: nms_bev, nms_normal_bev, boxes_iou_bev), all on srf_nms_bev / srf_iou_bev (csrc/nms_bev.cu).
Semantics restated from mmdet3d 1.0.0rc6 core/post_processing/box3d_nms.py and mmcv-full 1.7.0 ops/iou3d.py;
ties between equal scores keep the lower box index (the reference's sorts leave them unspecified).

`nms_device` is the graph-capturable core shared with SRFDetHead.nms_bboxes; the drop-ins read the kept count back
to the host, as their variable-length results require.
"""
import ctypes

import torch

from .. import _lib as L


def nms_device(boxes, scores, score_thr, iou_thr, rotated, max_num, post_center_range=None):
    """boxes (bs, k, dim >= 7) rows with x, y, dx, dy, yaw at columns 0, 1, 3, 4, 6; scores (bs, k, n_cls) fp32.
    -> device tensors out_boxes (bs, max_num, dim), out_scores (bs, max_num), out_labels / out_index (bs, max_num) int32,
    counts (bs,) int32; rows past the count: zero box, score 0, label / index -1.  No host synchronisation."""
    boxes, scores = boxes.float().contiguous(), scores.float().contiguous()
    bs, k, dim = boxes.shape
    n_cls = scores.shape[2]
    assert scores.shape[:2] == (bs, k), (boxes.shape, scores.shape)
    lib = L.load()
    need = lib.srf_nms_bev_ws_bytes(bs, k, n_cls)
    dev = boxes.device
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    ob = torch.empty((bs, max_num, dim), dtype=torch.float32, device=dev)
    osc = torch.empty((bs, max_num), dtype=torch.float32, device=dev)
    olab = torch.empty((bs, max_num), dtype=torch.int32, device=dev)
    oidx = torch.empty((bs, max_num), dtype=torch.int32, device=dev)
    cnt = torch.empty((bs,), dtype=torch.int32, device=dev)
    rng = L.f6(post_center_range) if post_center_range is not None else None
    L.check(lib.srf_nms_bev(L.ptr(boxes), bs, k, dim, L.ptr(scores), n_cls, float(score_thr), float(iou_thr), int(bool(rotated)),
                            int(max_num), rng, L.ptr(ws), ws.numel(), L.ptr(ob), L.ptr(osc), L.ptr(olab), L.ptr(oidx), L.ptr(cnt),
                            L.stream_ptr()), 'srf_nms_bev')
    return ob, osc, olab, oidx, cnt


def merge_aug_device(boxes, scores, labels, counts, views, n_cls, iou_thr, rotated, max_num):
    """srf_merge_aug_bev (mmdet3d merge_aug_bboxes_3d per sample): boxes (bs, A, m, dim), scores (bs, A, m), labels
    (bs, A, m) int32 and counts (bs, A) int32 of A views, views [(scale, horizontal, vertical)] in concatenation order.
    -> out_boxes (bs, max_num, dim), out_scores (bs, max_num), out_labels (bs, max_num) int32, counts (bs,) int32; rows past
    the count: zero box, score 0, label -1.  No host synchronisation."""
    boxes, scores = boxes.float().contiguous(), scores.float().contiguous()
    labels, counts = labels.int().contiguous(), counts.int().contiguous()
    bs, a, m, dim = boxes.shape
    assert scores.shape == labels.shape == (bs, a, m) and counts.shape == (bs, a) and len(views) == a
    lib = L.load()
    inv = (ctypes.c_float * a)(*[1.0 / float(s) for s, _, _ in views])      # fl32(1 / scale): Python double, then fp32
    flips = (ctypes.c_int32 * a)(*[(L.AUG_FLIP_HORIZONTAL if h else 0) | (L.AUG_FLIP_VERTICAL if v else 0) for _, h, v in views])
    need = ctypes.c_size_t(0)
    args = (bs, a, m, dim, inv, flips, int(n_cls), float(iou_thr), int(bool(rotated)), int(max_num))
    L.check(lib.srf_merge_aug_bev(None, None, None, None, *args, None, ctypes.byref(need), None, None, None, None, None),
            'srf_merge_aug_bev')
    dev = boxes.device
    ws = torch.empty(int(need.value), dtype=torch.uint8, device=dev)
    ob = torch.empty((bs, max_num, dim), dtype=torch.float32, device=dev)
    osc = torch.empty((bs, max_num), dtype=torch.float32, device=dev)
    olab = torch.empty((bs, max_num), dtype=torch.int32, device=dev)
    cnt = torch.empty((bs,), dtype=torch.int32, device=dev)
    L.check(lib.srf_merge_aug_bev(L.ptr(boxes), L.ptr(scores), L.ptr(labels), L.ptr(counts), *args, L.ptr(ws),
                                  ctypes.byref(ctypes.c_size_t(ws.numel())), L.ptr(ob), L.ptr(osc), L.ptr(olab), L.ptr(cnt),
                                  L.stream_ptr()), 'srf_merge_aug_bev')
    return ob, osc, olab, cnt


def xywhr2xyxyr(boxes_xywhr):
    """mmdet3d.core.bbox.xywhr2xyxyr: (N, 5) [x, y, w, h, r] -> [x1, y1, x2, y2, r]."""
    boxes = torch.zeros_like(boxes_xywhr)
    half_w, half_h = boxes_xywhr[..., 2] / 2, boxes_xywhr[..., 3] / 2
    boxes[..., 0] = boxes_xywhr[..., 0] - half_w
    boxes[..., 1] = boxes_xywhr[..., 1] - half_h
    boxes[..., 2] = boxes_xywhr[..., 0] + half_w
    boxes[..., 3] = boxes_xywhr[..., 1] + half_h
    boxes[..., 4] = boxes_xywhr[..., 4]
    return boxes


def _xyxyr_rows(boxes_xyxyr):
    """(N, 5) xyxyr -> (N, 7) rows [cx, cy, 0, dx, dy, 0, r] as mmcv converts them back (cx = (x1 + x2) / 2, dx = x2 - x1)."""
    b = boxes_xyxyr.float()
    rows = torch.zeros((b.shape[0], 7), dtype=torch.float32, device=b.device)
    rows[:, 0] = (b[:, 0] + b[:, 2]) / 2
    rows[:, 1] = (b[:, 1] + b[:, 3]) / 2
    rows[:, 3] = b[:, 2] - b[:, 0]
    rows[:, 4] = b[:, 3] - b[:, 1]
    rows[:, 6] = b[:, 4]
    return rows


def _single_class_nms(boxes, scores, thresh, rotated):
    n = boxes.shape[0]
    if n == 0:
        return torch.zeros((0,), dtype=torch.long, device=boxes.device)
    _, _, _, idx, cnt = nms_device(_xyxyr_rows(boxes)[None], scores.reshape(1, n, 1), float('-inf'), thresh, rotated, n)
    return idx[0, :int(cnt[0])].long()


def nms_bev(boxes, scores, thresh, pre_max_size=None, post_max_size=None):
    """mmcv.ops.nms_bev (mmcv 1.7): rotated NMS of (N, 5) xyxyr boxes -> kept indices in score order."""
    if pre_max_size is not None or post_max_size is not None:
        raise NotImplementedError('nms_bev: pre_max_size / post_max_size are not supported (box3d_multiclass_nms does not use them)')
    return _single_class_nms(boxes, scores, thresh, True)


def nms_normal_bev(boxes, scores, thresh):
    """mmcv.ops.nms_normal_bev (mmcv 1.7): axis-aligned NMS of (N, 5) xyxyr boxes (the angle is ignored)."""
    return _single_class_nms(boxes, scores, thresh, False)


def boxes_iou_bev(boxes_a, boxes_b):
    """mmcv.ops.boxes_iou_bev (mmcv 1.7): rotated BEV IoU of (M, 5) and (N, 5) xyxyr boxes -> (M, N)."""
    a, b = _xyxyr_rows(boxes_a), _xyxyr_rows(boxes_b)
    iou = torch.zeros((a.shape[0], b.shape[0]), dtype=torch.float32, device=a.device)
    L.check(L.load().srf_iou_bev(L.ptr(a), a.shape[0], 7, L.ptr(b), b.shape[0], 7, 1, L.ptr(iou), L.stream_ptr()), 'srf_iou_bev')
    return iou


def box3d_multiclass_nms(mlvl_bboxes, mlvl_bboxes_for_nms, mlvl_scores, score_thr, max_num, cfg, mlvl_dir_scores=None,
                         mlvl_attr_scores=None, mlvl_bboxes2d=None):
    """mmdet3d.core.post_processing.box3d_multiclass_nms (1.0.0rc6).  mlvl_bboxes (N, D), mlvl_bboxes_for_nms (N, 5) xyxyr,
    mlvl_scores (N, C + 1) with the background in the last column; cfg.use_rotate_nms / cfg.nms_thr.
    -> (bboxes (n, D), scores (n,), labels (n,) int64)."""
    if mlvl_dir_scores is not None or mlvl_attr_scores is not None or mlvl_bboxes2d is not None:
        raise NotImplementedError('box3d_multiclass_nms: direction / attribute scores and 2-D boxes are not supported')
    get = cfg.get if hasattr(cfg, 'get') else (lambda key, default=None: getattr(cfg, key, default))
    n, n_cls = mlvl_scores.shape[0], mlvl_scores.shape[1] - 1      # mmdet3d: the last column is the background
    dev = mlvl_bboxes.device
    if n == 0 or n_cls < 1:
        return (mlvl_bboxes.new_zeros((0, mlvl_bboxes.shape[-1])), mlvl_scores.new_zeros((0,)),
                torch.zeros((0,), dtype=torch.long, device=dev))
    rows = _xyxyr_rows(mlvl_bboxes_for_nms)[None]
    scores = mlvl_scores[:, :n_cls].float().contiguous()[None]
    _, osc, olab, oidx, cnt = nms_device(rows, scores, score_thr, get('nms_thr'), get('use_rotate_nms', True), max_num)
    m = int(cnt[0])
    idx = oidx[0, :m].long()
    return mlvl_bboxes[idx], osc[0, :m].to(mlvl_scores.dtype), olab[0, :m].long()
