"""Builds nerficg_b200/libnerf_b200.so with nvcc for sm_100a (cross-compiles without a GPU).

    python nerficg_b200/csrc/build.py [--force]

One object per .cu (compiled in parallel, rebuilt only when a source or header is newer),
linked into a single C-ABI shared library with the static CUDA runtime.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

CSRC = Path(__file__).resolve().parent
PKG = CSRC.parent
BUILD = CSRC / 'build'
LIB = PKG / 'libnerf_b200.so'
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '-Xcompiler', '-fPIC',
         '--expt-relaxed-constexpr', '-Xptxas', '-v']


def build(force: bool = False, verbose: bool = False) -> Path:
    BUILD.mkdir(exist_ok=True, parents=True)
    sources = sorted(CSRC.glob('*.cu'))
    headers = list(CSRC.glob('*.cuh')) + [PKG.parent / 'include' / 'nerf_b200.h']
    newest_header = max(h.stat().st_mtime for h in headers)

    def compile_one(src: Path):
        obj = BUILD / (src.stem + '.o')
        if not force and obj.exists() and obj.stat().st_mtime > max(src.stat().st_mtime, newest_header):
            return obj, ''
        r = subprocess.run([NVCC, *FLAGS, '-c', str(src), '-o', str(obj)], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}')
        (BUILD / (src.stem + '.ptxas.txt')).write_text(r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        results = list(ex.map(compile_one, sources))
    objs = [str(o) for o, _ in results]
    if verbose:
        for _, log in results:
            if log:
                print(log)
    if force or not LIB.exists() or any(Path(o).stat().st_mtime > LIB.stat().st_mtime for o in objs):
        r = subprocess.run([NVCC, '-shared', '-o', str(LIB), *objs, '-gencode', 'arch=compute_100a,code=sm_100a'],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
