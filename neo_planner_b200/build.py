"""Builds neo_planner_b200/libneoopt.so (hand-written sm_100a CUDA + the C ABI of include/neoopt.h) in-tree.

    python -m neo_planner_b200.build [--force] [-v]

nvcc cross-compiles without a GPU. The .so is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
SO = os.path.join(HERE, 'libneoopt.so')
SOURCES = ['neoopt.cu', 'test_prims.cu', 'device_api.cu']
DEPS = ['neoopt.cu', 'test_prims.cu', 'device_api.cu', 'libm_log.h', 'minco_tile.cuh', 'lbfgsb_tile.cuh', 'x87_nrm2.h', 'map_kernels.cuh', 'astar_warp.cuh', 'dd_exp.h', '../../include/neoopt.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-Wno-format-truncation', '-shared']


def nvcc_path() -> str:
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    return 'nvcc'


def stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return SO
    cmd = [nvcc_path(), *NVCC_FLAGS, *(['-Xptxas', '-v'] if verbose else []), '-o', SO,
           *[os.path.join(CSRC, s) for s in SOURCES]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return SO


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
