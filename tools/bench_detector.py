"""Detector-level timings (CUDA events on the launching stream, 512 MiB L2 flush between steps, median of `--iters`):

    python tools/bench_detector.py [--kinds nusc waymo] [--iters 20]

Per configuration (nusc_L, waymo_L; calibrated synthetic weights of RegionFeaturePipeline, production-size clouds,
the configs' rotated NMS on) one JSON line per case:
  simple_test B=1   graph replay + the read-back of the results to the host (latency, ms);
  infer B=1/2/4     one CUDA graph over the whole batch (frames/s);
  run_frames x4     RegionFeaturePipeline.run_frames: 4 single-frame graphs in flight on 4 streams (frames/s).
The first line names the GPU and its power limit.
"""
import argparse
import json
import os
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--kinds', nargs='+', default=['nusc', 'waymo'], choices=['nusc', 'waymo', 'kitti'])
    ap.add_argument('--iters', type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_detector.py needs a CUDA device')
    print(json.dumps(gpu_info()), flush=True)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device='cuda')
    for kind in a.kinds:
        bench_kind(kind, a.iters, flush)


if __name__ == '__main__':
    main()
