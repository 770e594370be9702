"""Build libpaacb.so (the C-ABI extension) in-tree with nvcc for sm_100a.

    python -m paac_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
gpurun snapshot.  cudart is linked statically so the library has no CUDA runtime dependency beyond
the driver; torch streams are driver-level handles and are passed through unchanged.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
ROOT = os.path.dirname(HERE)
OBJ_DIR = os.path.join(ROOT, 'build', 'paacb')
LIB = os.path.join(HERE, 'libpaacb.so')

NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
ARCH_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a']
CFLAGS = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr',
          '-Xptxas', '-v' if os.environ.get('PAACB_PTXAS_V') else '-warn-spills']


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _deps_mtime():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    hdrs.append(os.path.join(ROOT, 'include', 'paacb.h'))
    return max(os.path.getmtime(h) for h in hdrs)


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_m = _deps_mtime()
    jobs = []
    for src in sources():
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + '.o')
        stale = force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_m)
        jobs.append((src, obj, stale))

    def compile_one(job):
        src, obj, stale = job
        if not stale:
            return ''
        cmd = [NVCC] + ARCH_FLAGS + CFLAGS + ['-c', src, '-o', obj]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (src, r.stdout))
        return r.stdout

    with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
        outs = list(ex.map(compile_one, jobs))
    if verbose:
        for o in outs:
            if o.strip():
                print(o)
    objs = [j[1] for j in jobs]
    need_link = force or any(j[2] for j in jobs) or not os.path.exists(LIB)
    if need_link:
        cmd = [NVCC] + ARCH_FLAGS + ['-shared', '-cudart', 'static', '-o', LIB] + objs
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError('link failed:\n%s' % r.stdout)
    return LIB


if __name__ == '__main__':
    lib = build(force='--force' in sys.argv, verbose='--verbose' in sys.argv or True)
    print('built', lib, os.path.getsize(lib), 'bytes')
