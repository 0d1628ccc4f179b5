"""Pillar configs as whole detectors on CUDA: srf_pillar_encode_rows against the module chain srf_pillar_vfe ->
srf_pillars_scatter -> srf_nchw_to_rows bit for bit and against the oracle, the detector's infer against the composition
of its modules, batches against single clouds, graph capture (also through MultiSweepLoader) and tools/infer.py."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from srfdet_b200 import synth
from util import cuda, randomize_bn_, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VS, PC = [0.2, 0.2, 8], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
FLAG_SETS = {'new': dict(legacy=False), 'legacy': dict(legacy=True, with_distance=True), 'avg': dict(legacy=False, mode='avg')}
ENCODINGS = ['F32', 'BF16', 'F16', 'BF16X2', 'F16X2']


def _cfg(golden_dir, kind='model'):
    return os.path.join(golden_dir, 'configs', kind, 'srfdet_pillar_nusc_L.py')


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


# ------------------------------------------------------------------------------------------ kernel
def _blocks(counts, block_rows, t, c, ny, nx, seed):
    """Per-sample blocks as srf_hard_voxelize writes them: valid rows hold 1..t points with zero-padded slots and distinct
    cells (two of them off the grid); rows past a block's count hold garbage."""
    g = torch.Generator().manual_seed(seed)
    bs = len(counts)
    vox = torch.randn((bs, block_rows, t, c), generator=g) * 20.0
    num = torch.randint(-5, t + 5, (bs, block_rows), generator=g, dtype=torch.int32)
    coors = torch.randint(-3, max(ny, nx) + 3, (bs, block_rows, 4), generator=g, dtype=torch.int32)
    for b, n in enumerate(counts):
        n = max(0, min(n, block_rows))
        num[b, :n] = torch.randint(1, t + 1, (n,), generator=g, dtype=torch.int32)
        slot = torch.arange(t).view(1, t, 1)
        vox[b, :n] = vox[b, :n] * (slot < num[b, :n].view(n, 1, 1))
        cells = torch.randperm(ny * nx, generator=g)[:n]
        coors[b, :n] = torch.stack([torch.full_like(cells, b), torch.zeros_like(cells), cells // nx, cells % nx], 1).int()
        if n > 7:
            coors[b, 5, 2] = ny          # off the grid
            coors[b, 7, 3] = -1
    return cuda(vox), cuda(num), cuda(coors)


def _chain_rows(net, vox, num, coors, d_counts, ny, nx, enc):
    """The module chain: PillarFeatureNetCustom and PointPillarsScatter per block (each with its device count), then
    srf_nchw_to_rows (SRF_F32: the canvas as NHWC rows)."""
    from srfdet_b200 import _lib as L
    from srfdet_b200.plugin import PointPillarsScatter
    from srfdet_b200.plugin.bev_backbone import nchw_to_rows
    bs = vox.shape[0]
    cout = net.pfn_layers[0].units
    sc = PointPillarsScatter(cout, (ny, nx))
    canvas = torch.zeros((bs, cout, ny, nx), device='cuda')
    for b in range(bs):
        feats = net(vox[b], num[b], coors[b], num_voxels=d_counts[b:b + 1])
        sc.scatter_into(canvas, feats, coors[b], num_voxels=d_counts[b:b + 1])
    if enc == L.F32:
        return canvas.permute(0, 2, 3, 1).reshape(bs * ny * nx, cout)
    return nchw_to_rows(canvas, enc)[:bs * ny * nx]


COUNT_CASES = {'b1_empty': [0], 'b1_partial': [137], 'b1_full': [200], 'b1_above': [260], 'b1_negative': [-4],
               'b3_mixed': [0, 137, 260], 'b3_full_negative_partial': [200, -4, 50]}


@pytest.mark.parametrize('shape', [(20, 5), (1, 8)], ids=['T20_C5', 'T1_C8'])
@pytest.mark.parametrize('flags', list(FLAG_SETS))
@pytest.mark.parametrize('case', list(COUNT_CASES))
def test_encode_rows_equals_chain(case, flags, shape):
    """All five encodings: rows below B*ny*nx equal the chain's bit for bit (empty cells zero); rows past it untouched."""
    from srfdet_b200 import _lib as L
    from srfdet_b200.plugin import PillarFeatureNetCustom
    t, c = shape
    counts, block_rows, ny, nx = COUNT_CASES[case], 200, 40, 56
    torch.manual_seed(len(case) + 7 * t)
    net = PillarFeatureNetCustom(in_channels=c, feat_channels=[64], voxel_size=VS, point_cloud_range=PC, **FLAG_SETS[flags]).eval()
    randomize_bn_(net, 3)
    net = net.cuda()
    vox, num, coors = _blocks(counts, block_rows, t, c, ny, nx, seed=sum(map(ord, case)))
    d_counts = cuda(np.array(counts, np.int32))
    n = len(counts) * ny * nx
    w, b, fl = net._kernel_args(torch.device('cuda'))
    for name in ENCODINGS:
        enc = getattr(L, name)
        ref = _chain_rows(net, vox, num, coors, d_counts, ny, nx, enc)
        rows = net.encode_rows(vox, num, coors, d_counts, ny, nx, enc)
        assert rows.shape == ((n + 127) // 128 * 128, L.enc_width(enc, 64)) and rows.dtype == L.enc_torch_dtype(enc)
        assert torch.equal(_bits(rows[:n]), _bits(ref)), name
        # the same call into a caller's buffer: rows from n on are left as they were
        buf = torch.full((n + 64, L.enc_width(enc, 64)), 7.0, dtype=L.enc_torch_dtype(enc), device='cuda')
        L.check(L.load().srf_pillar_encode_rows(
            L.ptr(vox), L.ptr(num), L.ptr(coors), L.ptr(d_counts), len(counts), block_rows, t, c, L.ptr(w), L.ptr(b), 64,
            L.f3(VS), L.f3([net.x_offset, net.y_offset, net.z_offset]), fl, ny, nx, enc, L.ptr(buf), L.stream_ptr()),
            'srf_pillar_encode_rows')
        assert torch.equal(_bits(buf[:n]), _bits(ref)) and bool((buf[n:] == 7.0).all()), name
        valid = sum(max(0, min(k, block_rows)) for k in counts)
        nonzero = int((rows[:n] != 0).any(1).sum())
        assert nonzero <= valid and (valid == 0) == (nonzero == 0), name


def test_encode_rows_argument_checks():
    from srfdet_b200 import _lib as L
    lib = L.load()
    d = torch.zeros(4, dtype=torch.int32, device='cuda')
    w = torch.zeros(64 * 16, device='cuda')
    rows = torch.zeros(64, device='cuda')
    for t, c, cout, flags, enc in ((1025, 5, 64, 3, L.F16), (20, 9, 64, 3, L.F16), (20, 2, 64, 3, L.F16), (20, 5, 513, 3, L.F16),
                                   (20, 5, 64, 3, 5)):
        rc = lib.srf_pillar_encode_rows(L.ptr(w), L.ptr(d), L.ptr(d), L.ptr(d), 1, 1, t, c, L.ptr(w), L.ptr(w), cout, L.f3(VS),
                                        L.f3([0, 0, 0]), flags, 1, 1, enc, L.ptr(rows), L.stream_ptr())
        assert rc != 0 and b'srf_pillar_encode_rows' in lib.srf_last_error()


def test_encode_rows_vs_oracle(golden_dir):
    """Full-size nuScenes cloud through the detector's pillar_rows (hard voxelization into a block + the fused kernel)
    against O.hard_voxelize -> O.pillar_feature_net -> O.pillars_scatter, on fp32 rows."""
    from oracle import oracle as O
    from srfdet_b200 import _lib as L
    from srfdet_b200.plugin import SRFDetPointPath, load_config
    model = load_config(_cfg(golden_dir))['model']
    path = SRFDetPointPath(**{k: copy.deepcopy(model[k]) for k in ('pts_voxel_layer', 'pts_voxel_encoder', 'pts_middle_encoder')})
    torch.manual_seed(5)
    path.pts_voxel_encoder.pfn_layers[0].linear.reset_parameters()
    randomize_bn_(path, 6)
    pts = synth.cloud('nusc', 77)
    v, c, n, _ = O.hard_voxelize(pts, VS, PC, 20, 40000)
    coors = np.concatenate([np.zeros((len(c), 1), np.int32), c], 1)
    ref = O.pillar_feature_net({k: t.numpy() for k, t in path.pts_voxel_encoder.state_dict().items()}, v, n, coors, VS, PC,
                               legacy=False)
    ref_canvas = O.pillars_scatter(ref, coors, 1, 512, 512)
    rows, ny, nx = path.cuda().pillar_rows([cuda(pts)], L.F32)
    assert (ny, nx) == (512, 512) and len(c) > 20000
    got = rows[:ny * nx].view(ny, nx, 64).permute(2, 0, 1).cpu().numpy()
    np.testing.assert_allclose(got, ref_canvas[0], rtol=1e-5, atol=2e-5)


# ---------------------------------------------------------------------------------------- detector
def _seeded_detector(golden_dir, seed=11, kind='model'):
    from srfdet_b200.pipeline import init_synthetic_backbone, init_synthetic_head
    from srfdet_b200.plugin import SRFDet
    det = SRFDet.from_config(_cfg(golden_dir, kind))
    init_synthetic_backbone(det.pts_backbone, seed)
    init_synthetic_backbone(det.pts_neck, seed + 1)
    init_synthetic_head(det.bbox_head, seed + 2)
    randomize_bn_(det, seed + 3)
    return det.cuda()


@pytest.mark.parametrize('precision', ['fp16', 'fp32'])
def test_infer_equals_module_composition(golden_dir, precision):
    """infer (pillar_rows straight into the backbone) equals hard_padded -> PillarFeatureNetCustom -> PointPillarsScatter
    -> nchw_to_rows -> SECONDCustom.forward_rows -> FPN.forward_rows -> head -> nms_bboxes bit for bit."""
    from srfdet_b200.plugin.bev_backbone import _tc_enc, nchw_to_rows
    det = _seeded_detector(golden_dir)
    assert det.bbox_head.device_nms
    pts = cuda(synth.cloud('nusc', 43))
    got = [t.clone() for t in det.infer([pts], precision=precision)]
    o = det.pts_voxel_layer.hard_padded(pts, batch_idx=0)
    feats = det.pts_voxel_encoder(o['voxels'], o['num_points'], o['coors'], num_voxels=o['count'])
    canvas = det.pts_middle_encoder(feats, o['coors'], batch_size=1, num_voxels=o['count'])
    rows = nchw_to_rows(canvas, _tc_enc(precision))
    pyr = det.pts_neck.forward_rows(det.pts_backbone.forward_rows(rows, 1, 512, 512, precision), 1, precision)
    assert [tuple(p.shape) for p in pyr] == [(1, 128, 256 // 2 ** i, 256 // 2 ** i) for i in range(4)]
    logits, boxes = det.bbox_head(None, pyr, None, precision=precision)
    ref = det.bbox_head.nms_bboxes(logits, boxes)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
    assert int(got[3][0]) > 0


def test_batch_equals_single_clouds(golden_dir):
    """B = 2 in one call against two B = 1 calls: rows, canvas and FPN pyramid bit for bit; final rows at fp32 within
    1e-3 (the head's split-K reduction depends on the row count, as in test_batch_hard_voxel_equals_single_frames)."""
    from srfdet_b200 import _lib as L
    det = _seeded_detector(golden_dir)
    clouds = [cuda(synth.cloud('nusc', 50)), cuda(synth.cloud('nusc', 51, n_points=200000))]
    hw = 512 * 512
    for enc in (L.F16, L.BF16X2):
        rows2, _, _ = det.pillar_rows(clouds, enc)
        rows2 = rows2.clone()
        for i, c in enumerate(clouds):
            assert torch.equal(_bits(rows2[i * hw:(i + 1) * hw]), _bits(det.pillar_rows([c], enc)[0][:hw]))
    bev2 = det.extract_point_features(clouds)
    assert bev2.shape == (2, 64, 512, 512)
    pyr2 = [p.clone() for p in det.extract_pts_feat(clouds)]
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


def test_graph_replay_equals_eager(golden_dir):
    """One captured B = 2 infer, replayed on two different pairs of clouds, equals the eager result of each pair."""
    det = _seeded_detector(golden_dir)
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


def _loader_and_samples(golden_dir, bs, n_frames, seed):
    import sweep_oracle as SO
    from srfdet_b200.plugin import load_config
    from srfdet_b200.plugin import points as P
    steps = P.parse_test_pipeline(load_config(_cfg(golden_dir, 'pipeline'))['test_pipeline'])
    rng = np.random.default_rng(seed)
    samples = [SO.make_sample(rng, 20000 + 1500 * i, [20000 - 700 * (i + j) for j in range(10)]) for i in range(n_frames)]
    compact = [SO.merge(s, steps.load_dim, steps.use_dim, steps.sweeps, steps.point_cloud_range,
                        choices=P.choose_sweeps(len(s['sweeps']), steps.sweeps['sweeps_num'], steps.sweeps['test_mode']))
               for s in samples]
    return P.MultiSweepLoader(steps, batch_size=bs, max_points=25000), samples, compact


def test_loader_padded_equals_compact(golden_dir):
    """MultiSweepLoader's NaN-padded clouds (B = 2) give the compact clouds' outputs bit for bit: the NaN rows fall
    outside the range and form no pillar."""
    det = _seeded_detector(golden_dir, kind='pipeline')
    loader, samples, compact = _loader_and_samples(golden_dir, 2, 2, 31)
    loader.stage(samples)
    clouds, counts = loader()
    assert [int(k) for k in counts.cpu()] == [c.shape[0] for c in compact]
    got = [t.clone() for t in det.infer(clouds)]
    ref = det.infer([cuda(c) for c in compact])
    assert int(got[3].min()) > 0
    for a, b in zip(got, ref):
        assert torch.equal(a, b)


def test_one_graph_for_a_loader_sequence(golden_dir):
    """use_graph=True over 3 loader frames of different sizes: one captured graph, each replay equals the eager run."""
    det = _seeded_detector(golden_dir, kind='pipeline')
    loader, frames, _ = _loader_and_samples(golden_dir, 1, 3, 50)
    eager = []
    for s in frames:
        loader.stage([s])
        eager.append([t.clone() for t in det.infer(loader()[0])])
    det.use_graph = True
    for s, ref in zip(frames, eager):
        loader.stage([s])
        got = det.infer(loader()[0])
        for a, b in zip(got, ref):
            assert torch.equal(a, b)
    assert len(det._graphs) == 1
    assert not torch.equal(eager[0][0], eager[1][0])


@pytest.mark.parametrize('bs', [1, 2, 4])
def test_graph_batch_sizes(golden_dir, bs):
    """infer(use_graph=True) at B = 1, 2, 4 equals the eager call."""
    det = _seeded_detector(golden_dir)
    clouds = [cuda(synth.cloud('nusc', 100 + i, n_points=120000)) for i in range(bs)]
    ref = [t.clone() for t in det.infer(clouds)]
    det.use_graph = True
    got = det.infer(clouds)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
    assert len(det._graphs) == 1 and int(got[3].min()) > 0


def test_simple_test_and_tools_infer(golden_dir, tmp_path):
    """tools/infer.py with the pillar config, a saved seeded checkpoint and two .bin clouds equals an in-process
    simple_test of the same batch."""
    from srfdet_b200.plugin import SRFDet
    cfg = _cfg(golden_dir)
    src = _seeded_detector(golden_dir, seed=21)
    ckpt = str(tmp_path / 'pillar.pth')
    torch.save({'state_dict': {k: v.cpu() for k, v in src.state_dict().items()}, 'meta': {'epoch': 1}}, ckpt)
    files = []
    for s, n in ((90, None), (91, 80000)):
        p = str(tmp_path / f'cloud{s}.bin')
        synth.cloud('nusc', s, n_points=n).astype(np.float32).tofile(p)
        files.append(p)
    out = str(tmp_path / 'res.npz')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'), cfg, ckpt, '--points', *files, '--load-dim', '5',
                        '--precision', 'fp16', '--out', out], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert len([ln for ln in r.stdout.splitlines() if 'cloud9' in ln]) == 2
    det = SRFDet.from_config(cfg).cuda()
    det.load_checkpoint(ckpt)
    ref = det.simple_test([cuda(np.fromfile(f, dtype=np.float32).reshape(-1, 5)) for f in files], [{}, {}])
    got = np.load(out)
    assert len(ref) == 2 and ref[0]['pts_bbox']['scores_3d'].numel() > 0
    for i, r in enumerate(ref):
        for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
            np.testing.assert_array_equal(got[f'{i}.{k}'], r['pts_bbox'][k].numpy())
