"""Build libcbg_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

The shared library is git-ignored but travels to the GPU box with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.path.join(HERE, 'libcbg_b200.so')
SOURCES = ['api.cu', 'graph.cu', 'node_gemm.cu', 'node_gemm_tc.cu', 'node_gemm_f16.cu', 'edge.cu', 'x2h_tc.cu', 'misc.cu', 'batch.cu', 'ipa.cu', 'd3fg.cu']
HEADERS = ['cbg_common.cuh', 'cbg_kernels.cuh', 'cbg_layout.h', 'cbg_tc.cuh', '../../include/cbg_b200.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return 'nvcc'


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA source into cbgbench_b200/libcbg_b200.so. Returns the path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', LIB_PATH] + SOURCES
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError('nvcc failed building libcbg_b200.so')
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
