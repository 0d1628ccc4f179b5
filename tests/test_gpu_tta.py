"""Test-time augmentation on CUDA: srf_augment_points and srf_merge_aug_bev against aug_oracle bit for bit, and the
detector's infer_aug / aug_test against infer, against each other and against the oracle merge of the per-view results,
graph capture over a MultiSweepLoader sequence and tools/infer.py --info with the restated double-flip config."""
import ctypes
import itertools
import math
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

import aug_oracle as O
import nms_oracle
import sweep_oracle as SO
from srfdet_b200 import synth
from srfdet_b200.plugin import points as P
from srfdet_b200.plugin import registry
from util import cuda

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR = 0.4
FLIPS = list(itertools.product([False, True], repeat=2))
VIEWS = [(s, h, v) for s in (1.0, 0.95, 1.05) for h, v in FLIPS]
PCR = [-40.0, -40.0, -3.0, 40.0, 40.0, 1.0]


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


# ------------------------------------------------------------------------------------------ srf_augment_points
def _cloud(seed, n):
    """A nuScenes-like cloud plus points exactly on the range faces (before and after a flip)."""
    c = synth.cloud('nusc', seed, n_points=n).astype(np.float32)
    c[:8, :3] = np.float32([[40, 0, 0], [-40, 0, 0], [0, 40, 0], [0, -40, 0], [1, 1, 1], [1, 1, -3], [39.999, -39.999, 0.5],
                            [-40.0001, 5, 0]])
    return c


@pytest.mark.parametrize('use_range', [False, True])
@pytest.mark.parametrize('count', ['all', 'ragged', 'zero', 'padded'])
def test_augment_points_vs_oracle(use_range, count):
    """All four flip combinations at scales 1, 0.95 and 1.05 in one call: kept set, order and values bit for bit, NaN rows
    past each view's count; ragged and zero device counts with garbage past them; a NaN-padded loader cloud."""
    cap, n = 6000, {'all': 6000, 'ragged': 3777, 'zero': 0, 'padded': 4100}[count]
    cloud = _cloud(5, cap)
    if count == 'padded':
        cloud[n:] = np.nan
    rng = PCR if use_range else None
    d_count = None if count in ('all', 'padded') else cuda(np.int32([n]))
    out, counts = P.augment_points(cuda(cloud), VIEWS, rng, d_count)
    out, counts = out.cpu().numpy(), counts.cpu().numpy()
    assert out.shape == (len(VIEWS), cap, 5)
    src = cloud if count == 'padded' else cloud[:n]
    for a, view in enumerate(VIEWS):
        ref = O.augment_points(src, *view, rng)
        k = int(counts[a])
        assert k == ref.shape[0], (view, k, ref.shape)
        fin = ~np.isnan(ref).any(1)
        np.testing.assert_array_equal(_bits(out[a, :k][fin]), _bits(ref[fin]))
        assert np.isnan(out[a, :k][~fin]).any(1).all()
        assert np.isnan(out[a, k:]).all()
        if use_range:
            assert k < src.shape[0] or n == 0


def test_augment_points_argument_checks():
    from srfdet_b200 import _lib as L
    lib = L.load()
    pts = torch.zeros((10, 4), device='cuda')
    out = torch.zeros((1, 10, 4), device='cuda')
    cnt = torch.zeros(1, dtype=torch.int32, device='cuda')
    ws = torch.zeros(4096, dtype=torch.uint8, device='cuda')
    sz = ctypes.c_size_t(ws.numel())
    for n_cols, n_views, flips in ((2, 1, 0), (9, 1, 0), (4, 0, 0), (4, 33, 0), (4, 1, 4)):
        sc = (ctypes.c_float * max(n_views, 1))(*[1.0] * max(n_views, 1))
        fl = (ctypes.c_int32 * max(n_views, 1))(*[flips] * max(n_views, 1))
        rc = lib.srf_augment_points(L.ptr(pts), 10, n_cols, None, n_views, sc, fl, None, L.ptr(out), L.ptr(cnt), L.ptr(ws),
                                    ctypes.byref(sz), L.stream_ptr())
        assert rc == -1 and b'srf_augment_points' in lib.srf_last_error()


# ------------------------------------------------------------------------------------------ srf_merge_aug_bev
def _views_scene(seed, n_views, m, n_cls, dim=9, full=False):
    """Per-view NMS-like outputs (bs = 1) of one scene: boxes around shared centres in the original frame, put into each
    view's frame; counts 0..m (m for every view when full).  Re-drawn until no pair of mapped-back boxes has an oracle
    IoU within 1e-4 of THR, rotated or axis-aligned, so fp32 against float64 cannot flip a decision."""
    rng = np.random.default_rng(seed)
    views = [VIEWS[(3 + 5 * a) % len(VIEWS)] for a in range(n_views)]
    ctr = rng.uniform(-45, 45, (max(20, n_views * m // 12), 2))
    counts = np.full(n_views, m) if full else rng.integers(0, m + 1, n_views)
    if not full and n_views > 1:
        counts[0], counts[-1] = 0, m

    def draw(k, view):
        s, h, v = view
        b = np.zeros((k, dim), np.float32)
        b[:, :2] = ctr[rng.integers(0, len(ctr), k)] + rng.normal(0, 0.8, (k, 2))
        b[:, 2] = rng.uniform(-2, 0, k)
        b[:, 3] = rng.uniform(3.5, 4.8, k)
        b[:, 4] = rng.uniform(1.6, 2.1, k)
        b[:, 5] = rng.uniform(1.4, 1.8, k)
        b[:, 6] = rng.uniform(-math.pi, math.pi, k)
        b[:, 7:] = rng.normal(0, 1, (k, dim - 7))
        b[:, :6] *= np.float32(s)
        b[:, 7:] *= np.float32(s)
        if h:
            b[:, 1::7] *= -1
        if v:
            b[:, 0::7] *= -1
        return b
    boxes = np.zeros((n_views, m, dim), np.float32)
    for a in range(n_views):
        boxes[a] = draw(m, views[a])
    for _ in range(30):
        back = np.concatenate([O.bbox3d_mapping_back(boxes[a, :counts[a]], *views[a]) for a in range(n_views)])
        bad = np.zeros(len(back), bool)
        for rot in (True, False):
            bad |= (np.abs(nms_oracle.box_iou_bev(back, back, rot) - THR) < 1e-4).any(1)
        if not bad.any():
            break
        pos = np.nonzero(bad)[0]
        off = np.concatenate([[0], np.cumsum(counts)])
        for p in pos:
            a = int(np.searchsorted(off, p, side='right') - 1)
            boxes[a, p - off[a]] = draw(1, views[a])[0]
    assert not bad.any()
    total = int(counts.sum())
    scores = np.zeros((n_views, m), np.float32)
    perm = (rng.permutation(max(total, 1)) / max(total, 1) * 0.98 + 0.01).astype(np.float32)
    labels = np.full((n_views, m), -1, np.int32)
    k = 0
    for a in range(n_views):
        c = counts[a]
        scores[a, :c] = perm[k:k + c]
        labels[a, :c] = rng.integers(0, n_cls, c)
        k += c
    return boxes, scores, labels, counts.astype(np.int32), views


def _merge_gpu(boxes, scores, labels, counts, views, n_cls, rotated, max_num):
    from srfdet_b200.plugin.nms import merge_aug_device
    out = merge_aug_device(cuda(boxes), cuda(scores), cuda(labels), cuda(counts), views, n_cls, THR, rotated, max_num)
    return [t.cpu().numpy() for t in out]


def _check_merge(out, i, boxes, scores, labels, counts, views, rotated, max_num):
    ob, osc, olab, cnt = out
    res = [(boxes[a, :counts[a]], scores[a, :counts[a]], labels[a, :counts[a]]) for a in range(len(views))]
    rb, rs, rl, _ = O.merge_aug_bboxes_3d(res, views, THR, max_num, rotated)
    n = int(cnt[i])
    assert n == len(rb), (n, len(rb))
    np.testing.assert_array_equal(olab[i, :n], rl)
    np.testing.assert_array_equal(_bits(osc[i, :n]), _bits(rs))
    np.testing.assert_array_equal(_bits(ob[i, :n]), _bits(rb))
    assert (olab[i, n:] == -1).all() and (osc[i, n:] == 0).all() and (ob[i, n:] == 0).all()
    return n, int(sum(counts))


@pytest.mark.parametrize('n_cls', [1, 10])
@pytest.mark.parametrize('n_views,bs', [(1, 1), (2, 3), (4, 1), (8, 3)])
def test_merge_aug_vs_oracle(n_views, bs, n_cls):
    """Kept rows, labels, order and boxes bit for bit; view counts 0 through m; rotated and axis-aligned; max_num below
    and above the total."""
    m = 300
    scenes = [_views_scene(100 * n_views + 10 * n_cls + i, n_views, m, n_cls) for i in range(bs)]
    views = scenes[0][4]
    for sc in scenes:                       # one view list per call: the samples share it
        assert sc[4] == views
    stack = [np.stack([sc[j] for sc in scenes]) for j in range(4)]
    seen = set()
    for rotated in (True, False):
        for max_num in (40, 5000):
            out = _merge_gpu(*stack, views, n_cls, rotated, max_num)
            for i, sc in enumerate(scenes):
                n, total = _check_merge(out, i, *sc[:4], views, rotated, max_num)
                seen.add(n == max_num)
                assert n < total or total == 0 or n_views == 1
    assert seen == {True, False} or n_views == 1


def test_merge_aug_2400_in_one_class():
    """8 views x 300 rows, every row valid and of one class: 2400 candidates in one class segment."""
    boxes, scores, labels, counts, views = _views_scene(7, 8, 300, 1, full=True)
    assert int(counts.sum()) == 2400
    for rotated in (True, False):
        out = _merge_gpu(boxes[None], scores[None], labels[None], counts[None], views, 1, rotated, 5000)
        n, _ = _check_merge(out, 0, boxes, scores, labels, counts, views, rotated, 5000)
        assert 100 < n < 2400


def test_merge_aug_limits():
    from srfdet_b200 import _lib as L
    lib = L.load()
    need = ctypes.c_size_t(0)
    inv = (ctypes.c_float * 14)(*[1.0] * 14)
    fl = (ctypes.c_int32 * 14)(*[0] * 14)
    rc = lib.srf_merge_aug_bev(None, None, None, None, 1, 14, 300, 9, inv, fl, 10, THR, 1, 500, None, ctypes.byref(need),
                               None, None, None, None, None)
    assert rc == -3 and b'4096' in lib.srf_last_error()                  # 14 x 300 candidates: SRF_ERR_UNSUPPORTED
    rc = lib.srf_merge_aug_bev(None, None, None, None, 1, 13, 300, 9, inv, fl, 33, THR, 1, 500, None, ctypes.byref(need),
                               None, None, None, None, None)
    assert rc == -3
    rc = lib.srf_merge_aug_bev(None, None, None, None, 1, 13, 300, 9, inv, fl, 10, THR, 1, 500, None, ctypes.byref(need),
                               None, None, None, None, None)
    assert rc == 0 and need.value > 13 * 300 * 13 * 300 // 8


# ------------------------------------------------------------------------------------------ detector
def _det(golden_dir, name):
    if name == 'pillar':
        from test_gpu_pillar_detector import _seeded_detector
        det = _seeded_detector(golden_dir, kind='pipeline')
    else:
        from test_gpu_detector import _pipeline_and_detector
        _, det = _pipeline_and_detector(golden_dir, name)
    det.bbox_head.test_cfg['max_num'] = 500
    return det


def _resorted(out, i):
    boxes, scores, labels, counts = [t.cpu().numpy() for t in out]
    n = int(counts[i])
    order = np.lexsort((np.arange(n), -scores[i, :n].astype(np.float64)))
    return boxes[i, :n][order], scores[i, :n][order], labels[i, :n][order]


def _merged(out, i):
    boxes, scores, labels, counts = [t.cpu().numpy() for t in out]
    n = int(counts[i])
    return boxes[i, :n], scores[i, :n], labels[i, :n]


def _oracle_of_batch(out, bs, views):
    """aug_oracle.merge_aug_bboxes_3d of the per-view results of one (bs * A)-cloud batch, sample-major."""
    boxes, scores, labels, counts = [t.cpu().numpy() for t in out]
    res = []
    for i in range(bs):
        per = [(boxes[i * len(views) + a, :counts[i * len(views) + a]], scores[i * len(views) + a, :counts[i * len(views) + a]],
                labels[i * len(views) + a, :counts[i * len(views) + a]]) for a in range(len(views))]
        res.append(O.merge_aug_bboxes_3d(per, views, THR, 500))
    return res


NAMES = ['nusc_L', 'pillar', 'waymo_L']
DISTINCT = [(1.0, h, v) for h, v in FLIPS]


@pytest.mark.parametrize('name', NAMES)
def test_identity_view_equals_infer(golden_dir, name):
    """(a) infer_aug with the single identity view is infer re-sorted by (score desc, position asc).  Dynamic voxels
    (waymo) average with float atomics, so two runs differ in the last bits: compared in fp32 within 1e-3."""
    det = _det(golden_dir, name)
    kind = 'waymo' if name == 'waymo_L' else 'nusc'
    pts = cuda(synth.cloud(kind, 43, n_points=120000))
    prec = 'fp32' if name == 'waymo_L' else None
    ref = [t.clone() for t in det.infer([pts], precision=prec)]
    got = det.infer_aug([pts], [(1.0, False, False)] * 3, precision=prec)
    a, b = _resorted(ref, 0), _merged(got, 0)
    assert len(b[0]) > 0
    if name == 'waymo_L':
        assert abs(len(a[0]) - len(b[0])) <= 2
        k = min(len(a[0]), len(b[0]), 20)
        np.testing.assert_allclose(a[1][:k], b[1][:k], rtol=0, atol=1e-3)
        return
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize('name', NAMES)
def test_aug_test_infer_aug_and_oracle(golden_dir, name):
    """(b) aug_test on oracle-augmented clouds (B = 2, the 4 distinct flips) equals infer_aug on the original clouds, and
    (c) both equal aug_oracle's merge of the per-view results of that batch.  The batch is the comparison: per-view
    simple_test at B = 1 differs from a batch in the last bits of the head's split-K reduction
    (test_batch_hard_voxel_equals_single_frames).  nusc_L and pillar are bit for bit; waymo_L (float-atomic voxel
    means, two runs differ) checks (c) on one run's own per-view results and (b) on the merged scores within 1e-3."""
    from test_gpu_detector import _BoxType
    det = _det(golden_dir, name)
    kind = 'waymo' if name == 'waymo_L' else 'nusc'
    prec = 'fp32' if name == 'waymo_L' else None
    clouds = [synth.cloud(kind, 60 + i, n_points=90000 + 20000 * i) for i in range(2)]
    rng = PCR if name != 'waymo_L' else None
    got = [t.clone() for t in det.infer_aug([cuda(c) for c in clouds], DISTINCT, rng, precision=prec)]
    aug = [[cuda(O.augment_points(c, *v, rng)) for c in clouds] for v in DISTINCT]
    metas = [[dict(pcd_scale_factor=s, pcd_horizontal_flip=h, pcd_vertical_flip=v, box_type_3d=_BoxType) for _ in clouds]
             for s, h, v in DISTINCT]
    old = registry.get_precision()
    registry.set_precision(prec or old)
    try:
        res = det.forward_test(points=aug, img_metas=metas)
        batch = [t.clone() for t in det.infer([aug[a][i] for i in range(2) for a in range(4)])]
    finally:
        registry.set_precision(old)
    oracle = _oracle_of_batch(batch, 2, DISTINCT)
    assert len(res) == 2
    for i in range(2):
        r = res[i]['pts_bbox']
        assert isinstance(r['boxes_3d'], _BoxType) and r['labels_3d'].dtype == torch.int64
        bx, sc, lb = r['boxes_3d'].tensor.numpy(), r['scores_3d'].numpy(), r['labels_3d'].numpy()
        gb, gs, gl = _merged(got, i)
        assert len(sc) > 0
        if name == 'waymo_L':
            k = min(len(sc), len(gs), 20)
            np.testing.assert_allclose(sc[:k], gs[:k], rtol=0, atol=1e-3)
            continue
        np.testing.assert_array_equal(bx, gb)
        np.testing.assert_array_equal(sc, gs)
        np.testing.assert_array_equal(lb, gl)
        ob, os_, ol, _ = oracle[i]
        np.testing.assert_array_equal(bx, ob)
        np.testing.assert_array_equal(sc, os_)
        np.testing.assert_array_equal(lb, ol)
    if name == 'waymo_L':                   # (c) on the per-view results of one run
        from srfdet_b200.plugin.nms import merge_aug_device
        b, s, l, c = batch
        merged = merge_aug_device(b.view(2, 4, *b.shape[1:]), s.view(2, 4, -1), l.view(2, 4, -1), c.view(2, 4), DISTINCT,
                                  det.bbox_head.num_classes, THR, True, 500)
        for i in range(2):
            for x, y in zip(_merged(merged, i), oracle[i][:3]):
                np.testing.assert_array_equal(x, y)


def test_duplicated_views_equal_distinct(golden_dir):
    """infer_aug drops duplicate views; the full 8-view double-flip list through aug_test's undeduplicated merge of the
    same per-view results gives the same rows."""
    from srfdet_b200.plugin.nms import merge_aug_device
    det = _det(golden_dir, 'nusc_L')
    aug = P.parse_test_augmentations(registry.load_config(os.path.join(golden_dir, 'configs', 'pipeline',
                                                                       'srfdet_nusc_L_tta.py'))['test_pipeline'])
    pts = cuda(synth.cloud('nusc', 70, n_points=100000))
    got = [t.clone() for t in det.infer_aug([pts], aug.views, aug.view_range)]
    views = [cuda(O.augment_points(pts.cpu().numpy(), *v, aug.view_range)) for v in P.distinct_views(aug.views)]
    b, s, l, c = det.infer(views)
    idx = [P.distinct_views(aug.views).index(v) for v in aug.views]
    full = merge_aug_device(b[idx][None], s[idx][None], l[idx][None], c[idx][None], aug.views, det.bbox_head.num_classes,
                            THR, True, 500)
    for x, y in zip(_merged(full, 0), _merged(got, 0)):
        np.testing.assert_array_equal(x, y)


def _tta_samples(rng, n_frames, base=20000):
    return [SO.make_sample(rng, base + 1500 * i, [base - 700 * (i + j) for j in range(10)]) for i in range(n_frames)]


def test_one_graph_for_a_loader_sequence(golden_dir):
    """(d) use_graph=True over 3 MultiSweepLoader frames with the double-flip config's views and range: one captured
    graph, each replay equal to the eager run of its frame."""
    det = _det(golden_dir, 'nusc_L')
    aug = P.parse_test_augmentations(registry.load_config(os.path.join(golden_dir, 'configs', 'pipeline',
                                                                       'srfdet_nusc_L_tta.py'))['test_pipeline'])
    loader = P.MultiSweepLoader(aug.loader_steps, batch_size=1, max_points=25000)
    frames = _tta_samples(np.random.default_rng(50), 3)
    eager = []
    for s in frames:
        loader.stage([s])
        clouds, counts = loader()
        eager.append([t.clone() for t in det.infer_aug(clouds, aug.views, aug.view_range, counts=counts)])
    det.use_graph = True
    for s, ref in zip(frames, eager):
        loader.stage([s])
        clouds, counts = loader()
        got = det.infer_aug(clouds, aug.views, aug.view_range, counts=counts)
        for a, b in zip(got, ref):
            assert torch.equal(a, b)
    assert len(det._graphs) == 1
    assert not torch.equal(eager[0][0], eager[1][0]) and int(eager[0][3][0]) > 0


def test_tools_infer_info_tta(golden_dir, tmp_path):
    """(e) tools/infer.py --info with the double-flip config on synthetic infos equals an in-process infer_aug of the
    oracle's merged clouds, frame by frame."""
    from srfdet_b200.plugin import SRFDet
    from test_gpu_sweeps import _oracle, _steps
    cfg = os.path.join(golden_dir, 'configs', 'pipeline', 'srfdet_nusc_L_tta.py')
    torch.manual_seed(6)
    src = SRFDet.from_config(cfg)
    ckpt = str(tmp_path / 'model.pth')
    torch.save({'state_dict': src.state_dict()}, ckpt)
    samples = _tta_samples(np.random.default_rng(61), 2, base=15000)
    infos = []
    for i, s in enumerate(samples):
        def put(arr, sub, name):
            d = tmp_path / 'data' / sub / 'LIDAR_TOP'
            d.mkdir(parents=True, exist_ok=True)
            np.asarray(arr, np.float32).tofile(str(d / name))
            return f'./data/nuscenes/{sub}/LIDAR_TOP/{name}'
        sweeps = [dict(sw, data_path=put(sw['data_path'], 'sweeps', f'{i}_{j}.bin')) for j, sw in enumerate(s['sweeps'])]
        infos.append(dict(lidar_path=put(s['lidar_path'], 'samples', f'{i}.bin'), timestamp=s['timestamp'], sweeps=sweeps))
    pkl = str(tmp_path / 'infos.pkl')
    with open(pkl, 'wb') as f:
        pickle.dump(dict(infos=infos), f)
    out = str(tmp_path / 'res.npz')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'), cfg, ckpt, '--info', pkl, '--index', '0', '1',
                        '--data-root', str(tmp_path / 'data'), '--max-points', '17000', '--out', out],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    det = SRFDet.from_config(cfg).cuda()
    det.load_checkpoint(ckpt)
    aug = P.parse_test_augmentations(registry.load_config(cfg)['test_pipeline'])
    got = np.load(out)
    for i, s in enumerate(samples):
        merged = _oracle(s, _steps())        # the key frame and sweeps merged, range applied (symmetric range, 1.0 scale)
        ref = _merged(det.infer_aug([cuda(merged)], aug.views, aug.view_range), 0)
        for k, x in zip(('boxes_3d', 'scores_3d', 'labels_3d'), ref):
            np.testing.assert_array_equal(got[f'{i}.{k}'], x)
