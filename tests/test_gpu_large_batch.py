"""Large LiDAR batches on CUDA: srf_gemv_f32 past 8 rows (the DPG projections, one row per sample), the one-sequence
srf_hard_voxelize_batch against B separate srf_hard_voxelize calls, and the detector at B = 12 / 16 and with TTA batches
of more than 8 views."""
import ctypes
import os

import numpy as np
import pytest
import torch

import sweep_oracle as SO
from srfdet_b200 import _lib as L
from srfdet_b200 import synth
from util import cuda

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------ srf_gemv_f32
def _gemv(x, w, bias, relu):
    m, k = x.shape
    n = w.shape[0]
    out = torch.full((m, n), 7.0, device='cuda')
    L.check(L.load().srf_gemv_f32(L.ptr(x), m, k, L.ptr(w), n, L.ptr(bias), int(relu), L.ptr(out), L.stream_ptr()),
            'srf_gemv_f32')
    return out


@pytest.mark.parametrize('k,n', [(529, 1024), (1024, 3600)])
@pytest.mark.parametrize('m', [1, 7, 8, 9, 16, 33, 64])
def test_gemv_rows_equal_single_row_calls(m, k, n):
    """Every row of an m-row call is bit-identical to the 1-row call on that row (so the rows of a batch of any size
    equal the rows of the batch-1 DPG), and within fp32 rounding of a float64 product."""
    g = torch.Generator().manual_seed(m * 7 + k)
    x = cuda(torch.randn((m, k), generator=g))
    w = cuda(torch.randn((n, k), generator=g) / k ** 0.5)
    b = cuda(torch.randn((n,), generator=g))
    for bias in (None, b):
        for relu in (False, True):
            got = _gemv(x, w, bias, relu)
            for r in range(m):
                assert torch.equal(got[r], _gemv(x[r:r + 1].contiguous(), w, bias, relu)[0]), (r, bias is None, relu)
            xd, wd = x.double().cpu(), w.double().cpu()
            ref = xd @ wd.T + (0 if bias is None else bias.double().cpu())
            if relu:
                ref = ref.clamp_min(0)
            bound = (xd.abs() @ wd.abs().T + (0 if bias is None else bias.double().cpu().abs())) * (k * 2.0 ** -24) + 1e-30
            assert bool(((got.double().cpu() - ref).abs() <= bound).all())


# ------------------------------------------------------------------------------------------ srf_hard_voxelize_batch
T_PTS, MAX_VOX = 10, 20000
SENT_F, SENT_I = -1234.5, -777


def _geom():
    g = synth.GEOM['nusc']
    return L.make_geom(g['voxel_size'], g['pc_range'])


def _outputs(bs, c, want_voxels, want_mean):
    return dict(voxels=torch.full((bs, MAX_VOX, T_PTS, c), SENT_F, device='cuda') if want_voxels else None,
                num_points=torch.full((bs, MAX_VOX), SENT_I, dtype=torch.int32, device='cuda'),
                coors=torch.full((bs, MAX_VOX, 4), SENT_I, dtype=torch.int32, device='cuda'),
                mean=torch.full((bs, MAX_VOX, c), SENT_F, device='cuda') if want_mean else None,
                count=torch.full((bs,), SENT_I, dtype=torch.int32, device='cuda'))


def _batch_args(clouds):
    bs = len(clouds)
    return (ctypes.c_void_p * bs)(*[p.data_ptr() for p in clouds]), (ctypes.c_int32 * bs)(*[p.shape[0] for p in clouds])


def _batched(clouds, c, want_voxels, want_mean):
    lib, geom = L.load(), _geom()
    ptrs, ns = _batch_args(clouds)
    ws = torch.empty(lib.srf_hard_voxelize_batch_ws_bytes(ns, len(clouds), T_PTS, MAX_VOX), dtype=torch.uint8, device='cuda')
    o = _outputs(len(clouds), c, want_voxels, want_mean)
    L.check(lib.srf_hard_voxelize_batch(ptrs, ns, len(clouds), c, ctypes.byref(geom), T_PTS, MAX_VOX, L.ptr(o['voxels']),
                                        L.ptr(o['coors']), L.ptr(o['num_points']), L.ptr(o['mean']), L.ptr(o['count']),
                                        L.ptr(ws), ws.numel(), L.stream_ptr()), 'srf_hard_voxelize_batch')
    return o


def _singles(clouds, c, want_voxels, want_mean):
    """B srf_hard_voxelize calls, cloud b with batch_idx = b into block b of sentinel-filled outputs."""
    lib, geom = L.load(), _geom()
    o = _outputs(len(clouds), c, want_voxels, want_mean)
    for b, p in enumerate(clouds):
        ws = torch.empty(max(lib.srf_hard_voxelize_ws_bytes(p.shape[0], T_PTS, MAX_VOX), 1), dtype=torch.uint8, device='cuda')
        L.check(lib.srf_hard_voxelize(L.ptr(p), p.shape[0], c, ctypes.byref(geom), T_PTS, MAX_VOX, b,
                                      L.ptr(None if o['voxels'] is None else o['voxels'][b]), L.ptr(o['coors'][b]),
                                      L.ptr(o['num_points'][b]), L.ptr(None if o['mean'] is None else o['mean'][b]), None,
                                      L.ptr(o['count'][b:b + 1]), L.ptr(ws), ws.numel(), L.stream_ptr()), 'srf_hard_voxelize')
    return o


def _assert_blocks_equal(got, ref):
    """Whole outputs bit for bit (the same sentinels in both), and the sentinels past each block's count untouched."""
    for key in ('count', 'num_points', 'coors', 'voxels', 'mean'):
        a, b = got[key], ref[key]
        assert (a is None) == (b is None), key
        if a is not None:
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                               b.view(torch.int32) if b.dtype == torch.float32 else b), key
    counts = got['count'].cpu().tolist()
    for b, m in enumerate(counts):
        assert 0 <= m <= MAX_VOX
        assert bool((got['num_points'][b, m:] == SENT_I).all()) and bool((got['coors'][b, m:] == SENT_I).all())
        for key in ('voxels', 'mean'):
            if got[key] is not None:
                assert bool((got[key][b, m:] == SENT_F).all())
    return counts


def _ragged(bs, seed):
    """Clouds of 0 to 60000 points: cloud 0 is the largest and overflows MAX_VOX, cloud 1 (when bs > 1) is empty."""
    rng = np.random.default_rng(seed)
    sizes = [60000] + [0] * (bs > 1) + [int(v) for v in rng.integers(500, 16000, max(bs - 2, 0))]
    return [cuda(synth.cloud('nusc', seed * 100 + i, n_points=max(n, 1000))[:n]) for i, n in enumerate(sizes[:bs])]


@pytest.mark.parametrize('want', [(True, True), (False, True), (True, False), (False, False)],
                         ids=['voxels_mean', 'mean', 'voxels', 'neither'])
@pytest.mark.parametrize('bs', [1, 3, 9, 17])
def test_batch_voxelize_equals_single_calls(bs, want):
    clouds = _ragged(bs, 3 + bs)
    got, ref = _batched(clouds, 5, *want), _singles(clouds, 5, *want)
    counts = _assert_blocks_equal(got, ref)
    assert counts[0] == MAX_VOX                                        # the overflowing cloud is cut at max_voxels
    if bs > 1:
        assert counts[1] == 0
    if bs > 2:
        assert all(0 < m < MAX_VOX for m in counts[2:])


def test_batch_voxelize_nan_padded_loader_clouds(golden_dir):
    """MultiSweepLoader's fixed-capacity clouds: the NaN rows past each count stay out of range, in both paths."""
    from srfdet_b200.plugin import load_config
    from srfdet_b200.plugin import points as P
    steps = P.parse_test_pipeline(load_config(os.path.join(golden_dir, 'configs', 'pipeline', 'srfdet_nusc_L.py'))['test_pipeline'])
    rng = np.random.default_rng(17)
    samples = [SO.make_sample(rng, 9000 + 2500 * i, [9000 - 600 * (i + j) for j in range(10)]) for i in range(3)]
    loader = P.MultiSweepLoader(steps, batch_size=3, max_points=16000)
    loader.stage(samples)
    clouds, counts = loader()
    clouds = [p.clone() for p in clouds]
    c = clouds[0].shape[1]
    assert all(bool(torch.isnan(p[int(k):]).all()) for p, k in zip(clouds, counts.cpu())) and int(counts.min()) > 0
    got, ref = _batched(clouds, c, True, True), _singles(clouds, c, True, True)
    assert min(_assert_blocks_equal(got, ref)) > 0


def test_batch_voxelize_argument_checks():
    """Bad arguments return SRF_ERR_ARG before any launch."""
    lib, geom = L.load(), _geom()
    clouds = _ragged(3, 5)
    o = _outputs(3, 5, True, True)
    ptrs, ns = _batch_args(clouds)
    need = lib.srf_hard_voxelize_batch_ws_bytes(ns, 3, T_PTS, MAX_VOX)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    bad_geom = L.make_geom([0.075, 0.075, 0.2], [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0])
    bad_geom.vs[0] = 0.0

    def call(ptrs=ptrs, ns=ns, bs=3, c=5, g=geom, t=T_PTS, mv=MAX_VOX, coors=o['coors'], counts=o['count'], nbytes=need):
        return lib.srf_hard_voxelize_batch(ptrs, ns, bs, c, ctypes.byref(g), t, mv, L.ptr(o['voxels']), L.ptr(coors),
                                           L.ptr(o['num_points']), L.ptr(o['mean']), L.ptr(counts), L.ptr(ws), nbytes,
                                           L.stream_ptr())
    torch.cuda.synchronize()
    before = lib.srf_launch_count()
    negative = (ctypes.c_int32 * 3)(ns[0], -1, ns[2])
    null_cloud = (ctypes.c_void_p * 3)(ptrs[0], ptrs[1], None)      # cloud 1 is empty: a null pointer is fine there
    big = (ctypes.c_int32 * (L.HV_BATCH_MAX + 1))(*([1] * (L.HV_BATCH_MAX + 1)))
    cases = [dict(bs=0), dict(bs=L.HV_BATCH_MAX + 1, ns=big), dict(c=2), dict(c=9), dict(t=0), dict(mv=0), dict(ns=negative),
             dict(ptrs=null_cloud), dict(g=bad_geom), dict(coors=None), dict(counts=None), dict(nbytes=need - 1)]
    for kw in cases:
        assert call(**kw) == -1, kw            # SRF_ERR_ARG
    assert lib.srf_launch_count() == before
    assert bool((o['count'] == SENT_I).all()) and bool((o['coors'] == SENT_I).all())
    assert lib.srf_hard_voxelize_batch_ws_bytes(negative, 3, T_PTS, MAX_VOX) == 0
    assert lib.srf_hard_voxelize_batch_ws_bytes(ns, 0, T_PTS, MAX_VOX) == 0
    assert call() == 0


# ------------------------------------------------------------------------------------------ detector
def _chained_rows_agree(got, ref, tol=1e-3, max_frac=0.1):
    """Decoded rows of the five chained stages, B > 1 against B = 1, per proposal as in test_gpu_fusion_batch: the
    DynamicConv output projection picks its split-K from the row count (plugin/head.py:_linear), so later stages differ
    in the last bits, and the chained stages amplify that for a few proposals.  Most rows within tol of max |ref|, and a
    tiny median."""
    g = got.cpu().numpy().reshape(got.shape[0], -1).astype(np.float64)
    r = ref.cpu().numpy().reshape(ref.shape[0], -1).astype(np.float64)
    err = np.abs(g - r).max(1) / max(np.abs(r).max(), 1e-12)
    assert (err > tol).mean() <= max_frac and np.median(err) < 1e-4, ((err > tol).mean(), float(np.median(err)), float(err.max()))


def _clouds(bs, seed):
    return [cuda(synth.cloud('nusc', seed + i, n_points=60000 + 4000 * i)) for i in range(bs)]


def test_nusc_L_batch_12_equals_single_clouds(golden_dir):
    """nusc L at B = 12 (past the former 8-row limit of the DPG projections): the packed voxel lists equal the single
    clouds' bit for bit, and every sample's decoded rows agree with its B = 1 run under the per-proposal bound."""
    from test_gpu_detector import _pipeline_and_detector
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    clouds = _clouds(12, 300)
    mean, coors, total = det.voxelize_padded(clouds)
    off = 0
    for i, c in enumerate(clouds):
        o = det.pts_voxel_layer.hard_padded(c, batch_idx=i, want_voxels=False, want_mean=True)
        m = int(o['count'])
        assert torch.equal(coors[off:off + m], o['coors'][:m]) and torch.equal(mean[off:off + m], o['mean'][:m]), i
        off += m
    assert int(total) == off
    det.bbox_head.use_nms = False
    sc, bx = [t.clone() for t in det.infer(clouds, precision='fp32')]
    assert sc.shape[0] == 12
    for i, c in enumerate(clouds):
        sc1, bx1 = det.infer([c], precision='fp32')
        _chained_rows_agree(sc[i], sc1[0])
        _chained_rows_agree(bx[i], bx1[0])


def test_nusc_L_graph_replay_batch_12(golden_dir):
    """One captured B = 12 infer, replayed on two different sets of clouds, equals the eager result of each set."""
    from test_gpu_detector import _pipeline_and_detector
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    n = 50000
    sets = [[c[:n] for c in _clouds(12, s)] for s in (400, 500)]
    eager = [[t.clone() for t in det.infer(p)] for p in sets]
    det.use_graph = True
    for p, ref in zip(sets, eager):
        got = det.infer(p)
        for a, b in zip(got, ref):
            assert torch.equal(a, b)
    assert len(det._graphs) == 1
    assert not torch.equal(eager[0][0], eager[1][0]) and int(eager[0][3].min()) > 0


def test_pillar_batch_16_equals_single_clouds(golden_dir):
    """Pillar config at B = 16: voxel blocks and backbone input rows equal the single clouds' bit for bit; decoded rows
    under the per-proposal bound."""
    from test_gpu_pillar_detector import _bits, _seeded_detector
    det = _seeded_detector(golden_dir)
    clouds = _clouds(16, 600)
    blk = det.hard_voxel_blocks(clouds, want_voxels=True)
    for i, c in enumerate(clouds):
        o = det.pts_voxel_layer.hard_padded(c, batch_idx=i)
        m = int(o['count'])
        assert int(blk['count'][i]) == m > 0
        for key in ('voxels', 'num_points', 'coors'):
            assert torch.equal(blk[key][i, :m], o[key][:m]), (i, key)
    hw = 512 * 512
    rows, _, _ = det.pillar_rows(clouds, L.F16)
    rows = rows.clone()
    for i, c in enumerate(clouds):
        assert torch.equal(_bits(rows[i * hw:(i + 1) * hw]), _bits(det.pillar_rows([c], L.F16)[0][:hw])), i
    det.bbox_head.use_nms = False
    sc, bx = [t.clone() for t in det.infer(clouds, precision='fp32')]
    for i, c in enumerate(clouds):
        sc1, bx1 = det.infer([c], precision='fp32')
        _chained_rows_agree(sc[i], sc1[0])
        _chained_rows_agree(bx[i], bx1[0])


def _tta_det(golden_dir):
    from test_gpu_detector import _pipeline_and_detector
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    det.bbox_head.test_cfg['max_num'] = 500
    return det


def _merged_agree(got, ref):
    """Merged TTA results of a 12-view batch against a 4-view batch: the views run at different batch sizes, so the head's
    split-K differs (see _chained_rows_agree) and near-tied boxes may swap in the merge NMS: the counts agree within 2 and
    the leading scores within 1e-3."""
    n_got, n_ref = int(got[3]), int(ref[3])
    assert n_ref > 0 and abs(n_got - n_ref) <= 2, (n_got, n_ref)
    k = min(n_got, n_ref, 20)
    np.testing.assert_allclose(got[1][:k].cpu().numpy(), ref[1][:k].cpu().numpy(), rtol=0, atol=1e-3)


def test_infer_aug_three_clouds_four_views(golden_dir):
    """infer_aug with 3 clouds x the double-flip config's 4 distinct views (12 views in one batch) against three
    single-cloud infer_aug calls."""
    from srfdet_b200.plugin import points as P
    from srfdet_b200.plugin import registry
    det = _tta_det(golden_dir)
    aug = P.parse_test_augmentations(registry.load_config(os.path.join(golden_dir, 'configs', 'pipeline',
                                                                       'srfdet_nusc_L_tta.py'))['test_pipeline'])
    assert len(P.distinct_views(aug.views)) == 4
    clouds = _clouds(3, 700)
    got = [t.clone() for t in det.infer_aug(clouds, aug.views, aug.view_range)]
    assert got[0].shape[0] == 3
    for i, c in enumerate(clouds):
        ref = det.infer_aug([c], aug.views, aug.view_range)
        _merged_agree([t[i] for t in got], [t[0] for t in ref])


def test_infer_aug_nine_views_one_cloud(golden_dir):
    """One cloud with 9 distinct views (3 scales x 3 flips) runs as one 9-view batch."""
    det = _tta_det(golden_dir)
    views = [(s, h, v) for s in (0.95, 1.0, 1.05) for h, v in ((False, False), (True, False), (False, True))]
    out = det.infer_aug(_clouds(1, 800), views, [-40.0, -40.0, -3.0, 40.0, 40.0, 1.0])
    boxes, scores, labels, counts = out
    n = int(counts[0])
    assert 0 < n <= 500 and bool(torch.isfinite(boxes[0, :n]).all()) and bool((labels[0, :n] >= 0).all())
    assert bool((scores[0, :n - 1] >= scores[0, 1:n]).all())
