"""Micro-benchmarks of single C-ABI entry points at the production shapes of srfdet_voxel_nusc_LC
(CUDA events on the launching stream, 512 MiB L2 flush between iterations, median of `--iters`).

    python tools/bench_kernels.py [attention] [dwconv] [encoder] [nms] [frame_nms] [--iters 20]

Prints one JSON line per case: {"case", "us", "gbs" (algorithmic bytes / time), "bytes"}.
"""
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from srfdet_b200 import _lib as L   # noqa: E402


def timed(fn, iters, flush):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def report(case, us, nbytes=0, flops=0):
    print(json.dumps({'case': case, 'us': round(us, 2), 'gbs': round(nbytes / us / 1e3, 1) if nbytes else None,
                      'tflops': round(flops / us / 1e6, 2) if flops else None, 'bytes': nbytes}), flush=True)


def bench_attention(iters, flush):
    lib = L.load()
    for c, heads, n_p in [(128, 8, 900), (256, 8, 900)]:
        qkv = torch.randn(n_p, 3 * c, device='cuda')
        for name, enc in [('F32', L.F32), ('F16', L.F16), ('F16X2', L.F16X2)]:
            att = torch.empty((n_p, L.enc_width(enc, c)), dtype=L.enc_torch_dtype(enc), device='cuda')
            us = timed(lambda: L.check(lib.srf_mha_attention(L.ptr(qkv), 1, n_p, heads, c // heads, L.ptr(att), enc, L.stream_ptr()), 'attn'),
                       iters, flush)
            report(f'attention C{c} h{heads} P{n_p} out {name}', us, qkv.numel() * 4 + att.numel() * att.element_size(), 4 * n_p * n_p * c)


def bench_dwconv(iters, flush):
    lib = L.load()
    n, c = 6, 128
    x = None
    for lvl, (h, w) in enumerate([(232, 400), (116, 200), (58, 100)]):
        a = torch.randn(n, h, w, c, device='cuda').permute(0, 3, 1, 2)            # channels_last view
        ctot = c + (x.shape[1] if x is not None else 0)
        wt = torch.randn(ctot, 9, device='cuda')
        bias = torch.randn(ctot, device='cuda')
        ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
        buf = torch.empty((n, ho, wo, ctot), device='cuda')
        ma = L.map_view(a)
        mb = L.map_view(x) if x is not None else L.Map(None, 0, 0, 0, 0, 0)
        us = timed(lambda: L.check(lib.srf_dwconv3x3_s2(ctypes.byref(ma), ctypes.byref(mb), n, h, w, L.ptr(wt), L.ptr(bias), 1, 1, L.ptr(buf),
                                                        L.stream_ptr()), 'dw'), iters, flush)
        report(f'dwconv3x3_s2 level {lvl} ({n}x{ctot}x{h}x{w})', us, (n * h * w * ctot + buf.numel()) * 4)
        x = buf.permute(0, 3, 1, 2)


def bench_encoder(iters, flush):
    """Sparse-conv launches of one eagerly launched nusc_L frame (path scope), one kernel at a time: bench.py's
    kernel-family pass restricted to the encoder."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
    import bench
    from srfdet_b200 import synth
    from srfdet_b200.pipeline import RegionFeaturePipeline
    scope = os.environ.get('SRF_BENCH_SCOPE', 'path')          # 'full' adds the dense backbone / neck / head kernels
    pipe = RegionFeaturePipeline('nusc', fusion=False, precision=os.environ.get('SRF_PRECISION', 'fp16'), scope=scope)
    pts = torch.as_tensor(synth.cloud('nusc', 1000)).cuda()
    if scope == 'full':
        pipe.calibrate(torch.as_tensor(synth.cloud('nusc', 999)).cuda())
    fams, tot, layers = bench.kernel_families(pipe, pts, bench.peaks(), torch, reps=3)
    for f in fams:
        print(json.dumps({'case': f['family'], 'launches': f['launches'], 'us_per_launch': round(1e3 * f['ms'] / f['launches'], 2),
                          'ms': f['ms'], 'bound': f['bound'], 'frac': f['frac']}), flush=True)
    if os.environ.get('SRF_BENCH_CALLS'):
        for ms, name, fam in bench.kernel_families.per_call:
            if os.environ['SRF_BENCH_CALLS'] in fam or os.environ['SRF_BENCH_CALLS'] in name:
                print(json.dumps({'call': name, 'family': fam, 'us': round(ms * 1e3, 2)}))
    print(json.dumps({'case': 'encoder frame, serialised kernel time', 'ms': tot}))


def _full_pipe(kind, fusion, use_nms=False, use_graph=False):
    from srfdet_b200 import synth
    from srfdet_b200.pipeline import RegionFeaturePipeline
    pipe = RegionFeaturePipeline(kind, fusion=fusion, scope='full', use_nms=use_nms, use_graph=use_graph)
    pipe.calibrate(torch.as_tensor(synth.cloud(kind, 999)).cuda())
    return pipe


def bench_nms(iters, flush):
    """srf_nms_bev (IoU mask + per-class scans + merge) with the configs' settings (nms_thr 0.4, rotated, 300 per image,
    score_thr 0) on the decoded outputs of one real full frame: nusc (900 proposals, 10 classes), waymo (3 classes)."""
    from srfdet_b200 import synth
    from srfdet_b200.plugin.nms import nms_device
    for kind, fusion in [('nusc', True), ('waymo', False)]:
        pipe = _full_pipe(kind, fusion)
        pipe.run_frame(torch.as_tensor(synth.cloud(kind, 1000)).cuda())
        scores, boxes = pipe.last['scores'].contiguous(), pipe.last['det_boxes'].contiguous()
        cfg = pipe.head.test_cfg
        run = lambda: nms_device(boxes, scores, 0.0, 0.4, True, cfg['max_per_img'], cfg['post_center_range'])
        cnt = int(run()[-1][0])
        us = timed(run, iters, flush)
        bs, k, n_cls = scores.shape
        report(f'nms_bev {kind} bs{bs} P{k} cls{n_cls} (kept {cnt})', us, boxes.numel() * 4 + scores.numel() * 4)
        del pipe


def bench_frame_nms(iters, flush):
    """run_frames of the nusc_LC frame (CUDA graphs, 4 frames in flight) with use_nms off and on, alternated in one
    process; frames/s of each (L2 flushed before every step of 4 frames)."""
    from srfdet_b200 import synth
    clouds = [torch.as_tensor(synth.cloud('nusc', 1000 + i)).cuda() for i in range(4)]
    pipes = {tag: _full_pipe('nusc', True, use_nms=on, use_graph=True) for tag, on in [('off', False), ('on', True)]}
    ms = {tag: [] for tag in pipes}
    for rep in range(6):
        for tag, pipe in pipes.items():
            us = timed(lambda: pipe.run_frames(clouds), iters, flush)
            if rep:                                      # the first round captures the graphs
                ms[tag].append(us)
    for tag in pipes:
        us = sorted(ms[tag])[len(ms[tag]) // 2]
        print(json.dumps({'case': f'frame_nms nusc_LC run_frames x4, use_nms {tag}', 'us_per_step': round(us, 1),
                          'frames_per_s': round(4 / (us * 1e-6), 1)}), flush=True)


CASES = {'attention': bench_attention, 'dwconv': bench_dwconv, 'encoder': bench_encoder, 'nms': bench_nms, 'frame_nms': bench_frame_nms}

if __name__ == '__main__':
    iters = int(sys.argv[sys.argv.index('--iters') + 1]) if '--iters' in sys.argv else 20
    args = [a for i, a in enumerate(sys.argv[1:], 1) if not a.startswith('--') and sys.argv[i - 1] != '--iters']
    torch.cuda.set_device(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device='cuda')
    print(json.dumps({'gpu': torch.cuda.get_device_name(0)}), flush=True)
    for name in (args or list(CASES)):
        CASES[name](iters, flush)
