"""Multi-sweep point input on CUDA (srf_merge_sweeps through plugin/points.py's MultiSweepLoader): the kernel against the
numpy restatement bit for bit and against the literal rc6 transcription within 1 ulp, the detector on padded clouds
against the compact ones, one graph for a sequence of frames, and tools/infer.py --info."""
import ctypes
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

import sweep_oracle as O
from srfdet_b200.plugin import points as P
from srfdet_b200.plugin import registry
from test_gpu_detector import _pipeline_and_detector
from util import cuda, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NUSC_SWEEPS = dict(sweeps_num=10, load_dim=5, use_dim=[0, 1, 2, 3, 4], pad_empty_sweeps=True, remove_close=True,
                   test_mode=False)


def _steps(**sweeps):
    return P.PointSteps(5, [0, 1, 2, 3, 4], dict(NUSC_SWEEPS, **sweeps), O.NUSC_RANGE)


def _oracle(sample, steps, literal=False):
    sw = steps.sweeps
    if literal:
        return O.literal_pipeline(sample, steps.load_dim, steps.use_dim, sw, steps.point_cloud_range)
    choices = P.choose_sweeps(len(sample['sweeps']), sw['sweeps_num'], sw['test_mode']) if sw else None
    return O.merge(sample, steps.load_dim, steps.use_dim, sw, steps.point_cloud_range, choices=choices)


def _run(loader, samples):
    loader.stage(samples)
    clouds, counts = loader()
    return [c.cpu().numpy() for c in clouds], counts.cpu().numpy()


def _check_bitwise(cloud, count, ref):
    assert count == ref.shape[0]
    np.testing.assert_array_equal(cloud[:count].view(np.int32), ref.view(np.int32))
    assert np.isnan(cloud[count:]).all()


CASES = {
    'sweeps': dict(n=[[900, 1200, 0, 700, 1500], [400, 300]], sweeps={}),
    'sweeps_keep_close': dict(n=[[900, 1200, 0, 700]], sweeps=dict(remove_close=False)),
    'zero_sweeps_no_pad': dict(n=[[]], sweeps=dict(pad_empty_sweeps=False)),
    'pad_empty_remove_close': dict(n=[[], [500, 600]], sweeps={}),
    'pad_empty_keep_close': dict(n=[[]], sweeps=dict(remove_close=False)),
    'more_than_sweeps_num': dict(n=[[300] * 13], sweeps=dict(test_mode=True)),
}


@pytest.mark.parametrize('case', list(CASES))
def test_kernel_equals_oracle(case):
    """Same kept set, order, values and count as the float64 restatement, bit for bit, with edge points (|x| or |y|
    exactly 1, points exactly on range faces), empty sources and in-range garbage past every source count."""
    c = CASES[case]
    rng = np.random.default_rng(sorted(CASES).index(case))
    samples = [O.make_sample(rng, 1000 + 300 * i, n) for i, n in enumerate(c['n'])]
    steps = _steps(**c['sweeps'])
    loader = P.MultiSweepLoader(steps, batch_size=len(samples), max_points=2000)
    big = [O.make_sample(rng, 1990, [1990] * 10, edges=False) for _ in samples]
    _run(loader, big)                                     # fills the staging past the later counts
    loader._dev['files'][:, :, :, :3].fill_(3.0)          # ... and with in-range garbage
    clouds, counts = _run(loader, samples)
    for cl, n, s in zip(clouds, counts, samples):
        assert cl.shape == (11 * 2000, 5)
        _check_bitwise(cl, int(n), _oracle(s, steps))


def test_kernel_against_literal_transcription():
    """Against the literal rc6 code (numpy BLAS matmul): the same kept set, values within 1 float32 ulp."""
    rng = np.random.default_rng(21)
    steps = _steps()
    loader = P.MultiSweepLoader(steps, batch_size=1, max_points=40000)
    for n in ([30000] * 10, [20000, 0, 35000]):
        sample = O.make_sample(rng, 34000, n)
        clouds, counts = _run(loader, [sample])
        ref = _oracle(sample, steps, literal=True)
        got = clouds[0][:int(counts[0])]
        assert got.shape == ref.shape
        np.testing.assert_array_equal(got[:, 3:], ref[:, 3:])
        np.testing.assert_array_max_ulp(got[:, :3], ref[:, :3], maxulp=1)


def test_kernel_argument_checks():
    from srfdet_b200 import _lib as L
    lib = L.load()
    total = torch.zeros(1, dtype=torch.int32, device='cuda')
    cols = (ctypes.c_int32 * 5)(0, 1, 2, 3, 4)
    srcs = (L.SweepSrc * 1)(L.SweepSrc(0, 0, 4, L.SWEEP_TIME_LAG))
    rc = lib.srf_merge_sweeps(srcs, 1, None, None, None, cols, 5, None, 1.0, None, total.data_ptr(), None, 0, L.stream_ptr())
    assert rc == -1 and b'ld' in lib.srf_last_error()
    srcs = (L.SweepSrc * 1)(L.SweepSrc(0, 0, 5, 0))
    total.fill_(-1)
    L.check(lib.srf_merge_sweeps(srcs, 1, None, None, None, cols, 5, None, 1.0, None, total.data_ptr(), None, 0,
                                 L.stream_ptr()), 'merge')
    assert int(total) == 0


# ------------------------------------------------------------------------------------- detector
def _nusc_samples(rng, n_frames, base=20000):
    return [O.make_sample(rng, base + 1500 * i, [base - 700 * (i + j) for j in range(10)]) for i in range(n_frames)]


@pytest.mark.parametrize('bs', [1, 2])
def test_nusc_padded_equals_compact(golden_dir, bs):
    """nusc L (hard voxels): infer on the loader's NaN-padded clouds equals infer on the compact oracle clouds bit for
    bit, NMS rows included."""
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    steps = _steps()
    samples = _nusc_samples(np.random.default_rng(30 + bs), bs)
    loader = P.MultiSweepLoader(steps, batch_size=bs, max_points=25000)
    loader.stage(samples)
    clouds, counts = loader()
    got = [t.clone() for t in det.infer(clouds)]
    ref = det.infer([cuda(_oracle(s, steps)) for s in samples])
    assert int(got[3].min()) > 0
    for a, b in zip(got, ref):
        assert torch.equal(a, b)


def test_waymo_padded_within_tolerance(golden_dir):
    """waymo L (dynamic voxels, float-atomic voxel means): decoded outputs within the 1e-3 fp32 tolerance of the
    compact cloud."""
    _, det = _pipeline_and_detector(golden_dir, 'waymo_L')
    cfg = registry.load_config(os.path.join(golden_dir, 'configs', 'pipeline', 'srfdet_waymo_L.py'))
    steps = P.parse_test_pipeline(cfg['test_pipeline'])
    rng = np.random.default_rng(40)
    sample = O.make_sample(rng, 150000, [], load_dim=6)
    loader = P.MultiSweepLoader(steps, batch_size=1, max_points=160000)
    loader.stage([sample])
    clouds, counts = loader()
    ref_cloud = _oracle(sample, steps)
    assert int(counts[0]) == ref_cloud.shape[0]
    det.bbox_head.use_nms = False
    sc, bx = [t.clone() for t in det.infer(clouds, precision='fp32')]
    sc1, bx1 = det.infer([cuda(ref_cloud)], precision='fp32')
    assert rel_err(sc.cpu().numpy(), sc1.cpu().numpy()) < 1e-3
    assert rel_err(bx.cpu().numpy(), bx1.cpu().numpy()) < 1e-3


def test_one_graph_for_a_sequence(golden_dir):
    """use_graph=True over 3 frames of different sizes and poses through the loader: one captured graph, and each
    replay equals the eager run of its frame."""
    _, det = _pipeline_and_detector(golden_dir, 'nusc_L')
    steps = _steps()
    loader = P.MultiSweepLoader(steps, batch_size=1, max_points=25000)
    frames = _nusc_samples(np.random.default_rng(50), 3)
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


def test_tools_infer_info_end_to_end(golden_dir, tmp_path):
    """tools/infer.py --info on a synthetic infos pkl and .bin files equals an in-process simple_test of the oracle's
    merged clouds, frame by frame."""
    from srfdet_b200.plugin import SRFDet
    cfg = os.path.join(golden_dir, 'configs', 'pipeline', 'srfdet_nusc_L.py')
    torch.manual_seed(6)
    src = SRFDet.from_config(cfg)
    ckpt = str(tmp_path / 'model.pth')
    torch.save({'state_dict': src.state_dict()}, ckpt)
    rng = np.random.default_rng(60)
    samples = _nusc_samples(rng, 2, base=15000) + [O.make_sample(rng, 12000, [])]
    infos = []
    for i, s in enumerate(samples):
        def put(arr, sub, name):
            d = tmp_path / 'data' / sub / 'LIDAR_TOP'
            d.mkdir(parents=True, exist_ok=True)
            np.asarray(arr, np.float32).tofile(str(d / name))
            return f'./data/nuscenes/{sub}/LIDAR_TOP/{name}'
        sweeps = [dict(sw, data_path=put(sw['data_path'], 'sweeps', f'{i}_{j}.bin'), type='lidar')
                  for j, sw in enumerate(s['sweeps'])]
        infos.append(dict(lidar_path=put(s['lidar_path'], 'samples', f'{i}.bin'), timestamp=s['timestamp'],
                          sweeps=sweeps, token=f't{i}'))
    pkl = str(tmp_path / 'infos.pkl')
    with open(pkl, 'wb') as f:
        pickle.dump(dict(infos=infos, metadata=dict(version='v1.0-mini')), f)
    out = str(tmp_path / 'res.npz')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'), cfg, ckpt, '--info', pkl, '--index', '0',
                        '1', '2', '--data-root', str(tmp_path / 'data'), '--max-points', '17000', '--out', out],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert len([ln for ln in r.stdout.splitlines() if 'LIDAR_TOP' in ln]) == 3
    det = SRFDet.from_config(cfg).cuda()
    det.load_checkpoint(ckpt)
    got = np.load(out)
    for i, s in enumerate(samples):
        ref = det.simple_test([cuda(_oracle(s, _steps()))], [{}])[0]['pts_bbox']
        for k in ('boxes_3d', 'scores_3d', 'labels_3d'):
            np.testing.assert_array_equal(got[f'{i}.{k}'], ref[k].numpy())
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'infer.py'),
                        os.path.join(golden_dir, 'configs', 'model', 'srfdet_nusc_L.py'), ckpt, '--info', pkl],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode != 0 and 'test_pipeline' in r.stderr
