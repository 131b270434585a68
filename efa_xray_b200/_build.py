"""Build the CUDA library in-tree with nvcc for sm_100a.

    python -m efa_xray_b200._build        (or __graft_entry__.build())

Produces efa_xray_b200/csrc/libefa_xray_b200.so.  nvcc cross-compiles without a GPU.  The .so is
git-ignored but travels to the GPU box with the repo snapshot; nothing is JIT-compiled at run time.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc')
LIB = os.path.join(CSRC, 'libefa_xray_b200.so')
SOURCES = ['api.cu', 'setup.cu', 'obs_solve.cu', 'state_update.cu', 'state_update_mma.cu',
           'obs_solve_persistent.cu', 'obs_solve_dag.cu', 'state_sweep_2p.cu', 'relax.cu', 'interp.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def _stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, 'common.cuh'),
               os.path.join(os.path.dirname(os.path.dirname(CSRC)), 'include', 'efa_xray_b200.h')]
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace('.cu', '.o'))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', s, '-o', o]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed: %s\n%s\n%s' % (' '.join(cmd), r.stdout, r.stderr))
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for log in ex.map(run, jobs):
                if verbose and log:
                    print(log)
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs
        run(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
