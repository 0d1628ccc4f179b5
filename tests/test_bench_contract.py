"""bench.py's output contract, checked on the CPU: the reference arm (`--impl reference`, the restated CPU path on the host
cores) is run for one step and its JSON line carries every key the driver reads; the committed line of the B200 arm
(`profiles/r02_bench_nusc_LC.json`, written by `python bench.py` on a B200) carries the same contract plus `roofline`,
`kernels` and `cpu_baseline`; the reference arm never maps the product's CUDA library."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
             'data', 'config', 'e2e']


def _check_base(line):
    for k in BASE_KEYS:
        assert k in line, k
    assert line['metric'] == json.load(open(os.path.join(ROOT, 'BASELINE.json')))['metric'].split(' at ')[0]
    assert line['unit'] == 'frames/s' and line['higher_is_better'] is True and line['scaling'] == 'weak'
    assert line['vs_baseline'] is None                     # BASELINE.md holds no published number for this metric
    assert line['data'] == 'synthetic' and 'workload' in line['config'] and 'model' not in line['config']
    for k in ('value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'):
        assert k in line['e2e'], k


def test_reference_arm_line_and_isolation():
    code = ('import sys, runpy; sys.argv = ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"]\n'
            'try:\n    runpy.run_path(%r, run_name="__main__")\nexcept SystemExit:\n    pass\n'
            'sys.stderr.write("MAPPED=%%d\\n" %% ("libsrfdet_b200" in open("/proc/self/maps").read()))\n') % os.path.join(ROOT, 'bench.py')
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert 'MAPPED=0' in r.stderr                           # the CPU arm runs oracle/ only
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
    _check_base(line)
    assert line['impl'] == 'reference' and line['n_gpus'] == 1 and line['steps'] == 1
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0 and line['e2e']['value'] == line['value']
    cb = line['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == line['value'] and cb['sample']
    assert line['config']['workload'] == 'nusc_LC'


def test_dump_outputs_budget_and_fixed_sample(tmp_path):
    """--dump-outputs: float32 .npy per frame output, small arrays whole, large ones sampled at the same indices in every
    run, the directory within bench.DUMP_BYTES even at many frames in flight."""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location('bench_under_test', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    bev = torch.randn(1, 256, 184, 184, generator=g)                    # the nuScenes BEV map: 34.7 MB in float32
    result = torch.randn(900, 19, generator=g, dtype=torch.float64)
    for fif in (1, 4, 16):
        d = tmp_path / str(fif)
        bench.dump_outputs([(bev, result)] * fif, str(d))
        files = sorted(os.listdir(d))
        assert files == sorted(f'frame{j}_{n}.npy' for j in range(fif) for n in ('bev', 'result'))
        assert sum(os.path.getsize(d / f) for f in files) <= bench.DUMP_BYTES
        r = np.load(d / 'frame0_result.npy')
        assert r.dtype == np.float32 and np.array_equal(r, result.float().numpy())
        b = np.load(d / f'frame{fif - 1}_bev.npy')
        assert b.dtype == np.float32 and b.ndim == 1 and b.size < bev.numel()
        assert np.isin(b, bev.numpy()).all()
    bench.dump_outputs([(bev, result)] * 4, str(tmp_path / 'again'))
    assert np.array_equal(np.load(tmp_path / 'again' / 'frame3_bev.npy'), np.load(tmp_path / '4' / 'frame3_bev.npy'))


def test_committed_b200_line_contract():
    line = json.load(open(os.path.join(ROOT, 'profiles', 'r02_bench_nusc_LC.json')))
    _check_base(line)
    assert line['config']['workload'] == 'nusc_LC' and line['n_gpus'] == 1 and line['warmup'] >= 3
    assert line['gpu_launches'] == line['gpu_launches_per_frame'] * line['steps'] * line['config']['frames_per_step_per_gpu'] > 0
    assert line['e2e']['h2d_bytes_per_step'] > 0 and line['e2e']['d2h_bytes_per_step'] > 0 and line['e2e']['value'] < line['value']
    c = line['clocks']
    assert c['sm_mhz'] and c['sm_max_mhz'] and not set(c['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
    r = line['roofline']
    assert r['bound'] in ('hbm', 'tensor') and r['unit'] in ('GB/s', 'TFLOP/s')
    assert abs(r['frac'] - r['achieved'] / r['peak']) < 1e-3
    assert r['traffic'] is None or r['traffic'] > 0
    peaks = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks) and r['bound'] == 'hbm':
        assert abs(r['peak'] - json.load(open(peaks))['hbm_gbs']) < 1e-6       # the measured copy bandwidth is the denominator
    # achieved = algorithmic bytes per launch / launch time measured with CUDA events inside bench.py
    if r['bound'] == 'hbm':
        assert abs(r['achieved'] - r['algorithmic_bytes_per_launch'] / (r['launch_ms'] * 1e-3) / 1e9) / r['achieved'] < 0.02
    cb = line['cpu_baseline']
    assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['unit'] == 'frames/s' and cb['value'] > 0
    fam = {k['family'] for k in line['kernels']}
    for need in ('voxelize', 'rulebook build', 'sparse conv 32->32', 'BEV RoIAlign', 'image RoIAlign (6 cameras)', 'DynamicConv interaction'):
        assert need in fam, need
    assert all(0 <= k['frac'] <= 1.0 for k in line['kernels'])
