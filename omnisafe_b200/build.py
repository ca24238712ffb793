"""Build the C-ABI CUDA library (sm_100a) in-tree: omnisafe_b200/lib/libomnisafe_b200.so.

nvcc cross-compiles without a GPU; the built .so travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
INCLUDE = os.path.join(HERE, '..', 'include')
LIBDIR = os.path.join(HERE, 'lib')
LIB = os.path.join(LIBDIR, 'libomnisafe_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a',
    '-O3', '-lineinfo', '-std=c++17',
    '-Xcompiler', '-fPIC',
    '--expt-relaxed-constexpr',
]


def sources() -> list[str]:
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(('.cu', '.cuh', '.h'))]
    for path in files + [os.path.join(INCLUDE, 'omnisafe_b200.h')]:   # every source includes the C-ABI header
        with open(path, 'rb') as fh:
            h.update(os.path.basename(path).encode())
            h.update(fh.read())
    h.update(' '.join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, '.build_digest')
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp):
        with open(stamp) as fh:
            if fh.read().strip() == dig:
                return LIB
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(LIBDIR, os.path.basename(src)[:-3] + '.o')
        cmd = [NVCC, *FLAGS, '-I', INCLUDE, '-c', src, '-o', obj]
        if verbose:
            cmd.insert(1, '-Xptxas=-v')
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(out.decode())
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f'nvcc failed for {src}\n')
    if failed:
        raise RuntimeError('CUDA build failed')
    subprocess.check_call([NVCC, '-shared', '-o', LIB, *objs, '-lcudart'])
    with open(stamp, 'w') as fh:
        fh.write(dig)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
