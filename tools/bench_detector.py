"""Detector-level timings (CUDA events on the launching stream, 512 MiB L2 flush between steps, median of `--iters`):

    python tools/bench_detector.py [--kinds nusc waymo pillar] [--iters 20]

Per configuration (nusc_L, waymo_L; calibrated synthetic weights of RegionFeaturePipeline, production-size clouds,
the configs' rotated NMS on) one JSON line per case:
  simple_test B=1   graph replay + the read-back of the results to the host (latency, ms);
  infer B=1/2/4     one CUDA graph over the whole batch (frames/s);
  run_frames x4     RegionFeaturePipeline.run_frames: 4 single-frame graphs in flight on 4 streams (frames/s).
nusc_L also times the multi-sweep point input (plugin/points.py, synthetic key frame + 10 sweeps of about 35k points,
5 columns, random rigid poses, 8 frames of different point counts):
  merge kernel       srf_merge_sweeps alone at that shape (us per call, CUDA events, L2 flushed);
  sequence           infer B=1 with use_graph over the 8 frames from no captured graph, host clock to a device
                     synchronise: plain compact clouds (one capture per point count) vs the loader's fixed-capacity
                     clouds (stage + merge + one graph);
  replay             the same 8 frames again once every graph exists (median of --iters passes): the cost of voxelizing
                     over the capacity instead of the valid count, plus the loader's staging copies and merge.
pillar (the restated srfdet_pillar_nusc_L config, seeded synthetic weights, rotated NMS on):
  pillar kernel      srf_pillar_encode_rows against the chain it replaces (srf_pillar_vfe -> zeroed fp32 canvas +
                     srf_pillars_scatter -> srf_nchw_to_rows) on the same blocks, B = 1, a 300k-point nuScenes cloud
                     (up to 40000 pillars), fp16 rows; algorithmic bytes = pillars read (voxels, num_points, coors) +
                     rows written, GB/s against that;
  infer B=1/2/4      one CUDA graph over the batch, plain clouds and MultiSweepLoader clouds (stage + merge + graph).
The first line names the GPU and its power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def timed(fn, iters, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['power_limit_and_max_sm_clock'] = q
    except (OSError, subprocess.SubprocessError):
        info['power_limit_and_max_sm_clock'] = 'not available'
    return info


def bench_kind(kind, iters, flush):
    from srfdet_b200 import synth
    from srfdet_b200.pipeline import RegionFeaturePipeline, backbone_cfg, head_cfg, MODEL_CFG
    from srfdet_b200.plugin import SRFDet
    pipe = RegionFeaturePipeline(kind, fusion=False, scope='full', use_nms=True, use_graph=True)
    pipe.calibrate(torch.as_tensor(synth.cloud(kind, 44)).cuda())
    head = head_cfg(kind, False, use_nms=True)
    test_cfg = dict(pts=head.pop('test_cfg'))
    det = SRFDet(**MODEL_CFG[kind], **backbone_cfg(kind), bbox_head=head, test_cfg=test_cfg, use_graph=True).cuda()
    sd = dict(pipe.detector.state_dict())
    for prefix, m in (('pts_backbone.', pipe.backbone), ('pts_neck.', pipe.neck), ('bbox_head.', pipe.head)):
        sd.update({prefix + k: v for k, v in m.state_dict().items()})
    det.load_checkpoint(sd)
    clouds = [torch.as_tensor(synth.cloud(kind, 1000 + i)).cuda() for i in range(4)]
    name = f'{kind}_L'
    prec = pipe.precision

    def line(case, ms, frames):
        print(json.dumps(dict(config=name, case=case, precision=prec, ms=round(ms, 3), frames_per_s=round(frames / ms * 1e3, 1),
                              points=[int(c.shape[0]) for c in clouds[:frames]])), flush=True)
    line('simple_test B=1 (graph replay + read-back)', timed(lambda: det.simple_test(clouds[:1], [{}]), iters, flush), 1)
    for b in (1, 2, 4):
        line(f'infer B={b} (one graph)', timed(lambda: det.infer(clouds[:b]), iters, flush), b)
    line('run_frames x4 (4 single-frame graphs in flight)', timed(lambda: pipe.run_frames(clouds), iters, flush), 4)
    if kind == 'nusc':
        bench_sweeps(det, name, prec, iters, flush)


def _sweep_sample(rng, n_key, n_sweeps):
    """Synthetic nuScenes-like info: a ring cloud per file (synth.cloud), sweeps under random rigid poses 50 ms apart."""
    from srfdet_b200 import synth
    ts = 1533151603547590

    def pose():
        a = rng.uniform(-0.05, 0.05)
        return np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]), rng.normal(scale=2.0, size=3)
    sweeps = []
    for i, n in enumerate(n_sweeps):
        rot, trans = pose()
        sweeps.append(dict(data_path=synth.cloud('nusc', int(rng.integers(1 << 30)), n_points=n), sensor2lidar_rotation=rot,
                           sensor2lidar_translation=trans, timestamp=ts - 50000 * (i + 1)))
    return dict(lidar_path=synth.cloud('nusc', int(rng.integers(1 << 30)), n_points=n_key), timestamp=ts, sweeps=sweeps)


def _host_timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def bench_sweeps(det, name, prec, iters, flush):
    from srfdet_b200.plugin.points import MultiSweepLoader, PointSteps
    steps = PointSteps(5, [0, 1, 2, 3, 4], dict(sweeps_num=10, load_dim=5, use_dim=[0, 1, 2, 3, 4], pad_empty_sweeps=True,
                                                remove_close=True, test_mode=False), [-55.2, -55.2, -5.0, 55.2, 55.2, 3.0])
    loader = MultiSweepLoader(steps, batch_size=1, max_points=40000)
    rng = np.random.default_rng(7)
    frames = [_sweep_sample(rng, 34000 + 600 * f, [34500 - 300 * f - 200 * j for j in range(10)]) for f in range(8)]
    compact = []
    for smp in frames:
        loader.stage([smp])
        clouds, counts = loader()
        compact.append(clouds[0][:int(counts[0])].clone())

    def out(case, ms, frames_n, **extra):
        print(json.dumps(dict(config=name, case=case, precision=prec, ms=round(ms, 4),
                              frames_per_s=round(frames_n / ms * 1e3, 1) if frames_n else None, **extra)), flush=True)
    loader.stage([frames[0]])
    ms = timed(loader, iters * 5, flush)
    out('merge kernel (11 sources x ~35k points, 5 columns)', ms, 0, us_per_call=round(ms * 1e3, 1),
        input_rows=11 * 40000, kept_points=int(compact[0].shape[0]))

    def plain():
        for c in compact:
            det.infer([c])

    def staged():
        for smp in frames:
            loader.stage([smp])
            det.infer(loader()[0])
    det.reset_graphs()
    out('infer B=1 graph, sequence of 8 plain clouds (8 captures)', _host_timed(plain), 8, graphs=len(det._graphs),
        points=[int(c.shape[0]) for c in compact])
    rep = sorted(_host_timed(plain) for _ in range(iters))[iters // 2]
    out('infer B=1 graph, replay of 8 plain clouds (graphs exist)', rep, 8)
    det.reset_graphs()
    out('infer B=1 graph, sequence of 8 loader clouds (stage + merge, 1 capture)', _host_timed(staged), 8,
        graphs=len(det._graphs), capacity=loader.capacity)
    rep = sorted(_host_timed(staged) for _ in range(iters))[iters // 2]
    out('infer B=1 graph, replay of 8 loader clouds (stage + merge + one graph)', rep, 8)
    det.reset_graphs()


def bench_pillar(iters, flush):
    from srfdet_b200 import _lib as L
    from srfdet_b200 import synth
    from srfdet_b200.pipeline import init_synthetic_backbone, init_synthetic_head
    from srfdet_b200.plugin import SRFDet, load_config
    from srfdet_b200.plugin.bev_backbone import nchw_to_rows
    from srfdet_b200.plugin.points import MultiSweepLoader, parse_test_pipeline
    cfg = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'tests', 'golden', 'configs', 'pipeline',
                       'srfdet_pillar_nusc_L.py')
    det = SRFDet.from_config(cfg)
    init_synthetic_backbone(det.pts_backbone, 1)
    init_synthetic_backbone(det.pts_neck, 2)
    init_synthetic_head(det.bbox_head, 3)
    det = det.cuda()
    name, prec = 'pillar_nusc_L', 'fp16'

    def out(case, ms, frames_n, **extra):
        print(json.dumps(dict(config=name, case=case, precision=prec, ms=round(ms, 4),
                              frames_per_s=round(frames_n / ms * 1e3, 1) if frames_n else None, **extra)), flush=True)
    # ---- the kernel against the chain, on the same blocks
    cloud = torch.as_tensor(synth.cloud('nusc', 1000)).cuda()
    blk = det.hard_voxel_blocks([cloud], want_voxels=True)
    vfe, mid = det.pts_voxel_encoder, det.pts_middle_encoder
    ny, nx, enc = mid.ny, mid.nx, L.F16
    vox, num, coors, count = blk['voxels'], blk['num_points'], blk['coors'], blk['count']
    fused = lambda: vfe.encode_rows(vox, num, coors, count, ny, nx, enc)

    def chain():
        feats = vfe(vox[0], num[0], coors[0], num_voxels=count)
        return nchw_to_rows(mid(feats, coors[0], batch_size=1, num_voxels=count), enc)
    n_hw = ny * nx
    same = torch.equal(fused()[:n_hw].view(torch.int16), chain()[:n_hw].view(torch.int16))
    m = int(count[0])
    _, t, c = vox.shape[1:]
    bytes_fused = m * (t * c * 4 + 4 + 16) + n_hw * L.enc_width(enc, 64) * 2
    ms_f, ms_c = timed(fused, iters * 5, flush), timed(chain, iters * 5, flush)
    out('pillar kernel srf_pillar_encode_rows (B=1, fp16 rows)', ms_f, 0, us=round(ms_f * 1e3, 1), pillars=m,
        algorithmic_bytes=bytes_fused, gb_per_s=round(bytes_fused / ms_f / 1e6, 1), bit_identical_to_chain=same)
    out('pillar chain vfe -> zeroed fp32 canvas + scatter -> nchw_to_rows (B=1, fp16 rows)', ms_c, 0, us=round(ms_c * 1e3, 1),
        speedup_of_kernel=round(ms_c / ms_f, 2))
    # ---- the detector with one graph per batch shape
    det.use_graph = True
    clouds = [torch.as_tensor(synth.cloud('nusc', 1000 + i)).cuda() for i in range(4)]
    steps = parse_test_pipeline(load_config(cfg)['test_pipeline'])
    rng = np.random.default_rng(9)
    samples = [_sweep_sample(rng, 34000 + 600 * f, [34500 - 300 * f - 200 * j for j in range(10)]) for f in range(4)]
    for b in (1, 2, 4):
        out(f'infer B={b} (one graph, plain clouds)', timed(lambda: det.infer(clouds[:b]), iters, flush), b,
            points=[int(x.shape[0]) for x in clouds[:b]])
        loader = MultiSweepLoader(steps, batch_size=b, max_points=40000)

        def staged():
            loader.stage(samples[:b])
            det.infer(loader()[0])
        out(f'infer B={b} (one graph, loader clouds: stage + merge + graph)', timed(staged, iters, flush), b,
            capacity=loader.capacity)
    det.reset_graphs()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--kinds', nargs='+', default=['nusc', 'waymo', 'pillar'], choices=['nusc', 'waymo', 'kitti', 'pillar'])
    ap.add_argument('--iters', type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_detector.py needs a CUDA device')
    print(json.dumps(gpu_info()), flush=True)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device='cuda')
    for kind in a.kinds:
        if kind == 'pillar':
            bench_pillar(a.iters, flush)
        else:
            bench_kind(kind, a.iters, flush)


if __name__ == '__main__':
    main()
