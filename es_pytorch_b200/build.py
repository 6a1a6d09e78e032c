"""Build recipe for libes_b200.so (in-tree, sm_100a only).

``python -m es_pytorch_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles
without a GPU; the resulting .so is git-ignored but travels to the GPU box with the
repo snapshot.  cudart is linked statically so the library does not depend on which
libcudart torch happens to load.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libes_b200.so')
STAMP = os.path.join(HERE, '.libes_b200.stamp')

SOURCES = ['api.cu', 'reconstruct.cu', 'rank.cu', 'elementwise.cu', 'mt_draw.cu', 'mt_gauss.cu', 'rollout_f32.cu', 'rollout_f32x.cu', 'rollout_tc2.cu', 'rollout_tcw.cu', 'rollout_closed.cu']
HEADERS = ['common.cuh', 'tc_ptx.cuh', 'mt19937.cuh', 'mt_jump_polys.inc', os.path.join('..', '..', 'include', 'es_b200.h')]

NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a',
    '-O3', '-lineinfo', '-std=c++17',
    '--shared', '-Xcompiler', '-fPIC',
    '-cudart', 'static',
]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest() -> str:
    h = hashlib.sha256()
    for name in _sources() + HEADERS:
        with open(os.path.join(CSRC, name), 'rb') as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def nvcc_path() -> str:
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return 'nvcc'


def build_variant(name: str, defines) -> str:
    """Development: the same sources with extra -D flags -> es_pytorch_b200/libes_b200_<name>.so (load it with
    ES_B200_LIB=<path>; used by tools/ to time kernel variants side by side)."""
    out = os.path.join(HERE, f'libes_b200_{name}.so')
    cmd = [nvcc_path()] + NVCC_FLAGS + [f'-D{d}' for d in defines] + ['-o', out] + \
          [os.path.join(CSRC, s) for s in _sources()]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError('nvcc failed: ' + ' '.join(cmd))
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into es_pytorch_b200/libes_b200.so (no-op when up to date)."""
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == digest:
                return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + \
          ['-o', LIB] + [os.path.join(CSRC, s) for s in _sources()]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError('nvcc failed: ' + ' '.join(cmd))
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    with open(STAMP, 'w') as f:
        f.write(digest)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
