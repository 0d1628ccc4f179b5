#!/usr/bin/env python
"""bench.py -- frames/s of the SRFDet3D point-cloud -> region-feature hot path on B200.

  python bench.py --gpus N --steps K --warmup W [--workload nusc_LC|nusc_L|waymo_L|kitti_L]
                  [--scope full|path] [--precision fp16|fp32|bf16|fp32_simt] [--frames-in-flight F] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...          (one rank per GPU; frames are independent)
  python bench.py --impl reference ...        (restated reference CPU path on the host cores)

A step = a batch of F independent frames per rank (F = --frames-in-flight, default 4: BASELINE config 5's frame batches; every
frame is its own CUDA graph on its own stream, so latency-bound kernels of different frames overlap), each frame one pass of the hot path:
  scope 'full' (default): hard/dynamic voxelization (+VFE) -> SparseEncoder -> SECOND + FPN -> Dynamic Proposal
      Generation -> 5 CHAINED stages (BEV RoIAlign on the real FPN maps [+ 6-camera image RoIAlign + fusion Linear],
      self-attention, DynamicConv, FFN, towers, apply_deltas -> next stage's boxes) -> decode;
  scope 'path': the round-1 definition (voxelize -> SparseEncoder -> 5 stages of RoIAlign + DynamicConv on synthetic
      FPN maps and fixed boxes), kept for continuity.
`value` = frames/s over all ranks with the point clouds already resident in HBM;
`e2e` = the same through the public host-buffer call (pinned host points in, host results out, H2D + D2H inside
the timed region).  Prints ONE JSON line on rank 0; the extra objects are described in DESIGN.md 6:
`roofline` (dominant kernel), `kernels` (every kernel family of a frame, CUDA-event timed, with algorithmic
bytes / flops and roofline fraction), `modes` (other precision / scope / workload settings, including the
FP32-precision mode), `frames_in_flight_sweep` (BASELINE config 5 on one GPU), `cpu_baseline`.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    'nusc_L': dict(kind='nusc', fusion=False, desc='srfdet_voxel_nusc_L: 300k-pt 10-sweep nuScenes-shaped cloud, hard voxelization '
                   '0.075/0.075/0.2 m (1472x1472x41), 21-layer SparseEncoder, 900 proposals x 5 stages'),
    'nusc_LC': dict(kind='nusc', fusion=True, desc='srfdet_voxel_nusc_LC: nusc_L + 6-view image RoIAlign (1600x928 views, 4 FPN levels) + fusion Linear'),
    'waymo_L': dict(kind='waymo', fusion=False, desc='srfdet_dvoxel_waymo_L: 180k-pt cloud, dynamic voxelization + DynamicVFE'),
    'kitti_L': dict(kind='kitti', fusion=False, desc='srfdet_voxel_kitti_L: 120k-pt cloud, dynamic voxelization + DynamicVFE, C=256 head'),
}
SCOPES = {
    'full': 'voxelize -> SparseEncoder -> SECONDCustom + FPN -> DPG -> 5 chained stages (RoI sampling on the real FPN maps, attention, '
            'DynamicConv, FFN, towers, apply_deltas) -> decode',
    'path': 'voxelize -> SparseEncoder -> 5 stages of RoI sampling + DynamicConv on synthetic FPN maps and fixed boxes (round-1 definition)',
}
DTYPES = {'fp16': 'f16', 'bf16': 'bf16', 'fp32': 'f16x2 (hi+lo split operands on tcgen05, 3 MMAs per product, fp32 accumulate: FP32-mode tolerance 1e-4)',
          'fp32_simt': 'f32'}
N_CLOUDS = 8


def ncu_traffic():
    """family -> {dram_read_bytes_per_launch, dram_write_bytes_per_launch, ...} from the committed ncu --set full capture
    (profiles/r02_ncu_traffic.json, written by tools/ncu_summary.py traffic); {} when absent."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')) as f:
            return json.load(f)['families']
    except (OSError, ValueError, KeyError):
        return {}


TRAFFIC = ncu_traffic()
IMG_ROI_TOUCHED_BYTES = (TRAFFIC.get('image RoIAlign (6 cameras)') or {}).get('dram_read_bytes_per_launch')
METRIC = 'frames/s (voxelize+SparseEncoder+RoI fusion)'


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sust=d['bf16_tflops_sustained'], src='measured (MEASURED_PEAKS.json)')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src='fallback (B200_PROFILING.md)')


class ClockSampler:
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = f'/tmp/srf_clocks_{os.getpid()}.csv'

    def start(self):
        try:
            self.f = open(self.path, 'w')
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['no samples'])
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))


def kernel_families(pipe, pts, pk, torch, reps=3):
    """CUDA-event timing of every C-ABI call of one eagerly launched frame (events on the launching stream, a spin
    kernel hides the host's enqueue latency), grouped into kernel families with their ALGORITHMIC work."""
    from srfdet_b200 import _lib as L
    from srfdet_b200 import profiling
    enc = pipe.detector.pts_middle_encoder
    # one kernel at a time: the side streams of the timed frame (coarse-level geometry under the convolutions, image
    # branch under the encoder, parameter GEMM under the RoI sampler) are folded onto the main stream for this pass, so
    # every event pair brackets a kernel that has the GPU to itself
    saved = (enc.overlap_geometry, pipe.overlap_stage, pipe.overlap_image_branch)
    enc.overlap_geometry = pipe.overlap_stage = pipe.overlap_image_branch = False
    for _ in range(2):
        pipe._run_frame_eager(pts)
    best = None
    for _ in range(reps):
        enc.profile = []
        with profiling.capture() as cap:
            torch.cuda._sleep(60_000_000)
            pipe._run_frame_eager(pts)
            torch.cuda.synchronize()
        prof, enc.profile = enc.profile, None
        # sparse-conv work from the rulebooks, in call order
        sparse = []
        for e in prof:
            n_out, n_in = int(e['n_out']), int(e['n_in'])
            pairs = int((e['nbr'][:, :n_out] >= 0).sum())
            es_in, es_out = e['in_bytes'], e['out_bytes']
            sparse.append((2.0 * pairs * e['cin'] * e['cout'],
                           n_in * e['cin'] * es_in + n_out * e['cout'] * es_out + e['kvol'] * e['cin'] * e['cout'] * es_in + 4.0 * e['kvol'] * n_out,
                           dict(layer=e['layer'], n_in=n_in, n_out=n_out, pairs=pairs)))
        it = iter(sparse)

        def conv_work(s):
            if s['kvol'] == 9:                                      # dense BEV conv: every in-bounds neighbour is a pair
                rows = s['cap']
                es = profiling.ES[s['in_enc']]
                return 2.0 * rows * 9 * s['cin'] * s['cout'], s['in_rows'] * s['cin'] * es + rows * s['cout'] * profiling.ES[s['out_enc']] + 9 * s['cin'] * s['cout'] * es
            f, b, _ = next(it)
            return f, b
        n_vox = int(enc.last_counts[0])
        cnts = [int(c) for c in enc.last_counts]
        shapes = getattr(enc, 'last_level_shapes', None) or []
        ctx = dict(n_points=int(pts.shape[0]), c_points=int(pts.shape[1]), n_voxels=n_vox, conv_work=conv_work,
                   level_counts={d: c for (d, _), c in zip(shapes, cnts)}, cap_counts={cap: c for (_, cap), c in zip(shapes, cnts)},
                   img_roi_input_bytes=IMG_ROI_TOUCHED_BYTES)
        fams = profiling.families(cap, ctx, pk)
        tot = sum(f['ms'] for f in fams)
        if best is None or tot < best[0]:
            best = (tot, fams, sparse, list(cap.per_call))
    tot, fams, sparse, per_call = best
    enc.overlap_geometry, pipe.overlap_stage, pipe.overlap_image_branch = saved
    kernel_families.per_call = per_call
    for f in fams:
        f['share_of_kernel_time'] = round(f['ms'] / tot, 4)
    return fams, round(tot, 4), [dict(flops=f, bytes=b, **d) for f, b, d in sparse]


DUMP_BYTES = 64_000_000


def dump_outputs(frames_out, out_dir):
    """Writes what the caller of run_frame / run_frames receives for each frame j of one step, as float32
    out_dir/frame<j>_bev.npy (dense BEV map) and out_dir/frame<j>_result.npy (scope 'full': decoded boxes and class scores;
    scope 'path': region features).  An array larger than its equal share of DUMP_BYTES is stored as a sample of its
    flattened elements at seeded indices, the same in every run, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = (DUMP_BYTES // (2 * len(frames_out)) - 4096) // 4          # float32 elements per array (4 KB kept for the header)
    for j, arrays in enumerate(frames_out):
        for name, t in zip(('bev', 'result'), arrays):
            a = t.float().cpu().numpy()
            if a.size > share:
                a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
            np.save(os.path.join(out_dir, f'frame{j}_{name}.npy'), a)


def pipe_enc(pipe):
    from srfdet_b200 import _lib as L
    from srfdet_b200.plugin import registry
    e = registry.act_enc(pipe.precision)
    return L.F32 if e is None else e


def cpu_frame_seconds(state, kind, d, pts_np, torch):
    from oracle import cpu_pipeline
    from srfdet_b200 import synth
    t0 = time.perf_counter()
    cpu_pipeline.run_frame(state, kind, synth.GEOM[kind], d, pts_np)
    return time.perf_counter() - t0


CPU_SAMPLE = ('full frames through the oracle port of the reference CPU path (mmcv CPU voxelize loop in C, spconv native gather-mm-scatter '
              'with torch.mm, torch CPU conv2d backbone / neck, RoIAlign C loop over the host threads, torch CPU attention / linear / bmm / layer_norm)')


def run_reference(args, wl):
    """--impl reference: the restated reference CPU path (oracle) on the host cores, same workload and scope."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from oracle import oracle as O
    O.build_c()
    from srfdet_b200 import synth
    from srfdet_b200 import pipeline as P
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind = wl['kind']
    state = build_cpu_state(kind, wl['fusion'], args.scope)
    d = P.HEAD_CFG[kind]['d']
    clouds = [synth.cloud(kind, 1000 + i) for i in range(2)]
    warm = min(args.warmup, 2)          # a CPU frame takes seconds: keep the whole run within a few minutes
    for i in range(warm):
        cpu_frame_seconds(state, kind, d, clouds[i % 2], torch)
    t0 = time.perf_counter()
    for i in range(args.steps):
        cpu_frame_seconds(state, kind, d, clouds[i % 2], torch)
    dt = time.perf_counter() - t0
    fps = args.steps / dt
    line = dict(metric=METRIC, value=round(fps, 4), unit='frames/s', n_gpus=args.gpus, steps=args.steps, warmup=warm,
                ms_per_step=round(dt / args.steps * 1e3, 2), higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                data='synthetic', impl='reference',
                config=dict(workload=args.workload, scope=args.scope, description=wl['desc'], frames_per_step_per_gpu=1),
                cpu_baseline=dict(value=round(fps, 4), unit='frames/s', cores=cores, kind='port',
                                  sample=f'{args.steps} {CPU_SAMPLE}; {clouds[0].shape[0]} points per frame'),
                e2e=dict(value=round(fps, 4), unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def build_cpu_state(kind, fusion, scope):
    """Same seeded weights / synthetic maps as the GPU arm's pipeline, built on the host.  Constructing the
    modules does not load the CUDA library (srfdet_b200/_lib.py:make_geom is host arithmetic)."""
    from srfdet_b200.pipeline import RegionFeaturePipeline
    pipe = RegionFeaturePipeline(kind, fusion=fusion, device='cpu', precision='fp32', scope=scope)
    return pipe.state()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='nusc_LC', choices=sorted(WORKLOADS))
    ap.add_argument('--scope', default='full', choices=sorted(SCOPES))
    ap.add_argument('--precision', default='fp16', choices=sorted(DTYPES))
    ap.add_argument('--frames-in-flight', type=int, default=4,
                    help='frames per rank per step (BASELINE config 5: frame batches), each its own CUDA graph on its own stream')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the modes / sweep / kernel-family measurements (timed value and e2e only)')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel eagerly instead of replaying a CUDA graph of the frame')
    ap.add_argument('--nchw', action='store_true', help='path scope: RoI stage samples contiguous NCHW maps instead of channels_last')
    ap.add_argument('--profiler-range', action='store_true',
                    help='cudaProfilerStart/Stop around the device-resident timed steps (ncu --profile-from-start off: launch list of the timed region only)')
    ap.add_argument('--kernels-out', default=None, help='write the kernel-family table and the per-layer sparse-conv work (JSON) here')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the outputs of the last device-resident timed step to DIR/<name>.npy (float32, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == 'reference':
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    from srfdet_b200 import _lib as L
    from srfdet_b200 import frames, synth
    from srfdet_b200.pipeline import RegionFeaturePipeline
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (there is no CPU fallback)'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    lib = L.load()
    pk = peaks()
    kind = wl['kind']
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device='cuda')   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_pipe(workload, scope, precision):
        w = WORKLOADS[workload]
        pipe = RegionFeaturePipeline(w['kind'], fusion=w['fusion'], precision=precision, channels_last=not args.nchw, scope=scope)
        if scope == 'full':
            pipe.calibrate(torch.as_tensor(synth.cloud(w['kind'], 999)).cuda())
        return pipe

    def clouds_for(kind_):
        c = [synth.cloud(kind_, 1000 * (rank + 1) + i) for i in range(N_CLOUDS)]
        return c, [torch.as_tensor(x).cuda() for x in c], [torch.as_tensor(x).pin_memory() for x in c]

    def timed(pipe, inputs, steps, warmup, fif, host):
        """`steps` steps of `fif` concurrent frames; events on the current stream bracket each step; L2 flushed between.
        The per-frame outputs of the last step are left in timed.last."""
        def step(i):
            batch = [inputs[(i * fif + j) % N_CLOUDS] for j in range(fif)]
            if fif == 1 and not host:
                return [pipe.run_frame(batch[0])]
            elif fif == 1:
                return [pipe.run_frame_host(batch[0])]
            else:
                return pipe.run_frames(batch, host=host)
        for i in range(warmup):
            step(i)
        barrier()
        ranged = args.profiler_range and not host and pipe is timed.main_pipe
        if ranged:
            torch.cuda.cudart().cudaProfilerStart()
        evs = []
        for i in range(steps):
            flush.zero_()                                # evict the previous frames from L2 (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            timed.last = step(i)
            e1.record()
            evs.append((e0, e1))
        barrier()
        if ranged:
            torch.cuda.cudart().cudaProfilerStop()
            args.profiler_range = False                  # the first (headline) timed region only
        ms = sum(a.elapsed_time(b) for a, b in evs)
        return frames.max_over_ranks(ms, 'cuda')

    pipe = make_pipe(args.workload, args.scope, args.precision)
    timed.main_pipe = pipe
    clouds_np, clouds_dev, clouds_pin = clouds_for(kind)
    fif = max(1, args.frames_in_flight)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    pipe._run_frame_eager(clouds_dev[0])
    n0 = lib.srf_launch_count()
    pipe._run_frame_eager(clouds_dev[0])
    launches_per_frame = int(lib.srf_launch_count() - n0)      # this library's kernels per frame (counted eagerly)
    pipe.use_graph = not args.no_graph
    ms_dev = timed(pipe, clouds_dev, args.steps, args.warmup, fif, host=False)
    if args.dump_outputs and rank == 0:
        dump_outputs(timed.last, args.dump_outputs)     # before the end-to-end steps replay the same graphs
    ms_e2e = timed(pipe, clouds_pin, args.steps, args.warmup, fif, host=True)
    clocks = sampler.stop() if rank == 0 else None
    fps = world * args.steps * fif / (ms_dev * 1e-3)
    fps_e2e = world * args.steps * fif / (ms_e2e * 1e-3)
    out_bytes = int(pipe.run_frame(clouds_dev[0])[1].numel() * 4)

    kernels = roof = modes = sweep = cpu = None
    kernel_ms = None
    if rank == 0 and not args.no_extras:
        # ---- kernel families of one frame (eager, CUDA events per call)
        pipe.use_graph = False
        kernels, kernel_ms, sparse_layers = kernel_families(pipe, clouds_dev[0], pk, torch)
        pipe.use_graph = not args.no_graph
        if args.kernels_out:
            with open(args.kernels_out, 'w') as f:
                json.dump(dict(workload=args.workload, scope=args.scope, precision=args.precision, kernel_ms_per_frame=kernel_ms,
                               families=kernels, sparse_conv_layers=sparse_layers, calls_in_order=kernel_families.per_call), f, indent=1)
        # the dominant KERNEL: the largest family that is one kernel (one entry point) with algorithmic work attached
        single = [k for k in kernels if len(k['entry_points']) == 1 and (k['bytes'] > 0 or k['flops'] > 0)]
        dom = (single or kernels)[0]
        traffic, traffic_src = None, None
        t = TRAFFIC.get(dom['family'])
        if t:
            traffic = t['dram_read_bytes_per_launch'] + t['dram_write_bytes_per_launch']
            traffic_src = 'profiles/r02_ncu_traffic.json (ncu --set full, dram read+write per launch, cold cache)'
        n = dom['launches']
        roof = dict(bound=dom['bound'], kernel=f"{dom['family']} ({n} launches per frame; entry points {dom['entry_points']})",
                    achieved=dom['achieved'], peak=dom['peak'], unit=dom['unit'], frac=dom['frac'], traffic=traffic, traffic_source=traffic_src,
                    peak_source=f"{pk['src']} {'HBM copy bandwidth' if dom['bound'] == 'hbm' else 'bf16 sustained'}",
                    launch_ms=round(dom['ms'] / n, 4), algorithmic_flops_per_launch=dom['flops'] / n, algorithmic_bytes_per_launch=dom['bytes'] / n,
                    share_of_step_ms=dom['ms'], share_of_kernel_time=dom['share_of_kernel_time'],
                    note='dominant kernel family of the frame; every family is listed under "kernels"')
        # ---- other modes: the FP32-precision mode of the same workload, and the round-1 scope / LiDAR-only workload
        if world == 1:
            modes = {}
            for tag, (w_, s_, p_) in {'fp32 (reference precision, hi+lo split tcgen05)': (args.workload, args.scope, 'fp32'),
                                      'nusc_L full fp16': ('nusc_L', 'full', 'fp16'),
                                      'nusc_L path fp16 (round-1 definition)': ('nusc_L', 'path', 'fp16'),
                                      'nusc_LC path fp16 (round-1 definition)': ('nusc_LC', 'path', 'fp16')}.items():
                if (w_, s_, p_) == (args.workload, args.scope, args.precision):
                    continue
                p2 = make_pipe(w_, s_, p_)
                p2.use_graph = True
                _, cd, cp = (clouds_np, clouds_dev, clouds_pin) if WORKLOADS[w_]['kind'] == kind else clouds_for(WORKLOADS[w_]['kind'])
                st = max(10, args.steps // 2)
                m1 = timed(p2, cd, st, 3, fif, host=False)        # same frames in flight as the headline
                m2 = timed(p2, cp, st, 3, fif, host=True)
                modes[tag] = dict(workload=w_, scope=s_, precision=p_, frames_in_flight=fif, value=round(st * fif / (m1 * 1e-3), 2),
                                  e2e=round(st * fif / (m2 * 1e-3), 2), ms_per_step=round(m1 / st, 4), steps=st)
                del p2
                torch.cuda.empty_cache()
            # ---- frames in flight on one GPU (BASELINE config 5)
            sweep = {}
            for f_ in (1, 2, 4, 8):
                st = max(6, args.steps // 2)
                m1 = timed(pipe, clouds_dev, st, 3, f_, host=False)
                m2 = timed(pipe, clouds_pin, st, 3, f_, host=True)
                sweep[str(f_)] = dict(value=round(st * f_ / (m1 * 1e-3), 2), e2e=round(st * f_ / (m2 * 1e-3), 2))
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            state = pipe.state()
            cpu_frame_seconds(state, kind, pipe.d, synth.cloud(kind, 1, n_points=20000), torch)   # warm caches / build
            t = cpu_frame_seconds(state, kind, pipe.d, clouds_np[0], torch)
            cpu = dict(value=round(1.0 / t, 4), unit='frames/s', cores=cores, kind='port',
                       sample=f'1 {CPU_SAMPLE}; {clouds_np[0].shape[0]} points, {t:.1f} s')
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    n_pts, c_pts = clouds_np[0].shape
    line = dict(metric=METRIC, value=round(fps, 2), unit='frames/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=round(ms_dev / args.steps, 4), higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype=DTYPES[args.precision], data='synthetic',
                config=dict(workload=args.workload, scope=args.scope, description=wl['desc'], scope_description=SCOPES[args.scope],
                            frames_per_step_per_gpu=fif,
                            parallelism=f'{world} independent frame replica(s), no data-path collective',
                            l2='512 MiB flush written between timed steps; 8 distinct clouds cycled',
                            launch='eager' if args.no_graph else 'one CUDA graph per frame (captured once, replayed)',
                            weights='synthetic: seeded random init, BatchNorm2d statistics of the dense backbone / neck / DPG calibrated on one frame',
                            excluded='image backbone (VoVNet/FPN: the image branch samples synthetic image FPN maps), rotated NMS'),
                clocks=clocks,
                e2e=dict(value=round(fps_e2e, 2), unit='frames/s', h2d_bytes_per_step=int(n_pts * c_pts * 4 * fif),
                         d2h_bytes_per_step=out_bytes * fif, ms_per_step=round(ms_e2e / args.steps, 4)),
                gpu_launches=launches_per_frame * args.steps * fif,
                gpu_launches_per_frame=launches_per_frame,
                roofline=roof, kernels=kernels, kernel_ms_per_frame_eager=kernel_ms, modes=modes, frames_in_flight_sweep=sweep,
                cpu_baseline=cpu)
    print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
