"""Builds libsfmloss.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libsfmloss.so')
SOURCES = ['api.cu', 'plan.cu', 'prep.cu', 'smooth.cu', 'fused_loss.cu', 'full_res.cu', 'mean_norm.cu', 'stage.cu', 'ingest.cu', 'eval.cu', 'comm.cu']
HEADERS = ['common.cuh', 'kernels.h', 'ssim_march.cuh', 'min_reprojection.cuh', 'geometry.cuh', 'smooth_task.cuh', os.path.join(ROOT, 'include', 'sfmloss.h')]


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found')


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    cmd = [_nvcc(), '--threads', '0', '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
           '-Xcompiler', '-fPIC', '-shared', '-I', os.path.join(ROOT, 'include'), '-I', CSRC,
           '-o', LIB] + [os.path.join(CSRC, s) for s in SOURCES] + ['-ldl']
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + res.stdout)
    if verbose:
        print(res.stdout)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
