"""Build libsrfdet_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m srfdet_b200.build [--force]

The shared object is plain C ABI (include/srfdet_b200.h); it links only cudart.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
SO = os.path.join(CSRC, 'libsrfdet_b200.so')
SOURCES = ['index.cu', 'voxelize.cu', 'scatter.cu', 'spconv_simt.cu', 'igemm_umma.cu', 'spconv_warp16.cu', 'roi.cu', 'dynconv.cu', 'pillar.cu', 'head_tail.cu', 'bev_dense.cu', 'attention.cu', 'conv3x3_halo.cu', 'nms_bev.cu', 'sweeps.cu', 'augment.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-O2', '--expt-relaxed-constexpr']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return 'nvcc'


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(CSRC, 'common.cuh'), os.path.join(CSRC, 'igemm_common.cuh'),
                                                        os.path.join(HERE, '..', 'include', 'srfdet_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), so=SO):
    """defines/so: development variants (e.g. -DSRF_IGEMM_PROF -> libsrfdet_b200_prof.so, tools/igemm_prof.py)."""
    if not force and not defines and not needs_build():
        return so
    objs = []
    procs = []
    tag = '_' + os.path.basename(so).replace('libsrfdet_b200_', '').replace('.so', '') if defines else ''
    for s in SOURCES:
        obj = os.path.join(CSRC, s.replace('.cu', tag + '.o'))
        if defines and os.path.exists(os.path.join(CSRC, s.replace('.cu', '.o'))):
            text = open(os.path.join(CSRC, s)).read() + open(os.path.join(CSRC, 'igemm_common.cuh')).read() * (s == 'igemm_umma.cu')
            if not any(d.split('=')[0] in text for d in defines):
                objs.append(os.path.join(CSRC, s.replace('.cu', '.o')))      # this source does not see the variant's macros
                continue
        cmd = ([_nvcc()] + NVCC_FLAGS + ['-D' + d for d in defines] + (['-Xptxas', '-v'] if verbose else [])
               + ['-c', os.path.join(CSRC, s), '-o', obj])
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(f'--- {s}\n{out}\n')
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed')
    link = [_nvcc(), '-shared', '-o', so] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    subprocess.check_call(link)
    return so


if __name__ == '__main__':
    if '--variant' in sys.argv:      # python -m srfdet_b200.build --variant NAME MACRO=VALUE ...
        i = sys.argv.index('--variant')
        print(build(force=True, defines=tuple(sys.argv[i + 2:]), so=SO.replace('.so', '_' + sys.argv[i + 1] + '.so')))
    elif '--prof' in sys.argv:
        print(build(force=True, defines=('SRF_IGEMM_PROF=' + ('2' if '--stages' in sys.argv else '1'),), so=SO.replace('.so', '_prof.so')))
    else:
        print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
