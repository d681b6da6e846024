"""Builds babyai_b200/libbabyai_b200.so (the C-ABI library of include/babyai_b200.h)
from babyai_b200/csrc/pool.cu with nvcc for sm_100a, in-tree."""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'csrc', 'pool.cu')
# every source the library is compiled from: a change to any of them rebuilds it
DEPS = sorted(glob.glob(os.path.join(HERE, 'csrc', '*'))) + [os.path.join(HERE, '..', 'include', 'babyai_b200.h')]
OUT = os.path.join(HERE, 'libbabyai_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')


def build(force=False, verbose=False):
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    cmd = [NVCC, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
           '--fmad=false',           # the reward is float64 arithmetic that must round like CPython's
           '-Xcompiler', '-fPIC', '-shared', '-cudart', 'shared', SRC, '-o', OUT]
    if verbose:
        cmd.insert(1, '-Xptxas')
        cmd.insert(2, '-v')
    subprocess.check_call(cmd)
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
