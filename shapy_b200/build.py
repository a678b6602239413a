"""Builds shapy_b200/libshapy_b200.so in-tree with nvcc for sm_100a (no torch dependency).

    python -m shapy_b200.build [--force]

Each .cu is compiled to an object (in parallel, cached by mtime) and linked into one shared
library whose exported symbols are exactly the `extern "C"` entry points of include/shapy_b200.h.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
# experiment variants: SHAPY_BUILD_TAG=x SHAPY_BUILD_DEFS="-DFOO=1" builds libshapy_b200_x.so next to the default
# library (select it at run time with SHAPY_B200_LIB=<path>); the default build has neither set.
TAG = os.environ.get('SHAPY_BUILD_TAG', '')
DEFS = os.environ.get('SHAPY_BUILD_DEFS', '').split()
OBJ = os.path.join(HERE, '_obj' + ('_' + TAG if TAG else ''))
LIB = os.path.join(HERE, 'libshapy_b200' + ('_' + TAG if TAG else '') + '.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC',
          '--expt-relaxed-constexpr']
# per-file extra flags: the triangle predicates must round like the plain-C oracle
EXTRA = {'measure.cu': ['-fmad=false'], 'measure_grad.cu': ['-fmad=false'], 'bvh.cu': ['-fmad=false']}


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith('.cu'))


def _newest_header():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    hs.append(os.path.join(os.path.dirname(HERE), 'include', 'shapy_b200.h'))
    return max(os.path.getmtime(h) for h in hs)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr = _newest_header()
    jobs = []
    for f in sources():
        src = os.path.join(CSRC, f)
        obj = os.path.join(OBJ, f[:-3] + '.o')
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr):
            cmd = [NVCC] + ARCH + COMMON + DEFS + EXTRA.get(f, []) + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
            jobs.append((f, cmd))

    def run(job):
        f, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return f, r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for f, r in ex.map(run, jobs):
                if verbose or r.returncode:
                    sys.stderr.write(f'--- {f}\n{r.stdout}{r.stderr}\n')
                if r.returncode:
                    raise RuntimeError(f'nvcc failed on {f}')
    objs = [os.path.join(OBJ, f[:-3] + '.o') for f in sources()]
    if force or jobs or not os.path.exists(LIB):
        cmd = [NVCC] + ARCH + ['-shared', '-o', LIB] + objs + ['-lcudart_static', '-lpthread', '-ldl', '-lrt']
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError('link failed')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
