"""In-tree build of libmavd.so with nvcc for sm_100a (no torch headers: the library is plain C ABI)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
INCLUDE = os.path.join(os.path.dirname(HERE), 'include')
SOURCES = ['api.cu', 'farneback.cu', 'detect.cu', 'sparse.cu']
OUT = os.path.join(CSRC, 'libmavd.so')


def nvcc_path() -> str:
    for cand in (shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found')


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh'))]
    deps.append(os.path.join(INCLUDE, 'mavd.h'))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    cmd = [nvcc_path(), '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
           '-Xcompiler', '-fPIC', '-shared', '-I', INCLUDE, '--threads', '3', '-o', OUT] + \
          [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, '-Xptxas')
        cmd.insert(2, '-v')
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n%s\n%s' % (res.stdout, res.stderr))
    if verbose:
        print(res.stderr)
    return OUT


if __name__ == '__main__':
    print(build(force=True, verbose=True))
