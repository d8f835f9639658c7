"""Build the sm_100a shared library in-tree with nvcc (no torch extension machinery: the
library has a plain C ABI, see include/kwiiyatta_b200.h)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.path.join(HERE, 'libkwiiyatta_b200.so')
SOURCES = ['dtw.cu', 'gmm.cu', 'gmm_tc.cu', 'gmm_diagblocks.cu', 'convert.cu', 'assemble.cu',
           'capi.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '--threads', '0',
              '-shared', '-Xcompiler', '-fPIC']


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh')]
    deps.append(os.path.join(HERE, '..', 'include', 'kwiiyatta_b200.h'))
    return os.path.getmtime(LIB_PATH) < max(os.path.getmtime(d) for d in deps)


def build(force=False, verbose=False):
    if not force and not is_stale():
        return LIB_PATH
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', LIB_PATH] + sources()
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == '__main__':
    print(build(force=True, verbose=True))
