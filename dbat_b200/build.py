"""Build libdbatgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libdbatgpu.so')
SOURCES = ['eval.cu', 'schur.cu', 'schur_win.cu', 'chol.cu', 'tilechol.cu', 'tilesym.cu', 'plan.cu', 'general_io.cu', 'covstats.cu', 'api.cu',
           'startval.cu', 'order.cu']
EXTRA = os.environ.get('DBAT_NVCC_EXTRA', '').split()
NVCC_FLAGS = EXTRA + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC']


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    headers.append(os.path.join(HERE, '..', 'include', 'dbat_gpu.h'))
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace('.cu', '.o'))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', s, '-o', o]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode())
        if p.returncode:
            raise RuntimeError('nvcc failed: ' + ' '.join(cmd))
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-ldl']
        subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
