"""Builds libgen6d_b200.so in-tree with nvcc for sm_100a (no JIT cache, so the .so travels with
the repo snapshot to the GPU box).  `python -m gen6d_b200.build [--force] [-v]`"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libgen6d_b200.so')
STAMP = os.path.join(HERE, '.libgen6d_b200.hash')
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC']
NO_FMA = ('glue.cu', 'track.cu')


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest():
    h = hashlib.sha256()
    files = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h')))
    files.append(os.path.join(os.path.dirname(HERE), 'include', 'gen6d_b200.h'))
    for f in files:
        h.update(f.encode())
        h.update(open(f, 'rb').read())
    h.update(' '.join(NVCC_FLAGS + list(NO_FMA)).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ and link the shared library.  Returns the library path."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read() == dig:
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + '.o')
        objs.append(obj)
        extra = ['-fmad=false'] if os.path.basename(src) in NO_FMA else []      # numpy-like rounding (glue_math.cuh)
        cmd = [nvcc] + NVCC_FLAGS + extra + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f'--- {os.path.basename(src)}\n{out}\n')
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed building libgen6d_b200.so')
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-lcudart']
    subprocess.run(cmd, check=True)
    with open(STAMP, 'w') as f:
        f.write(dig)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
