"""Builds libdrb.so (the C-ABI library, include/drb.h) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the snapshot."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libdrb.so')
SOURCES = ['api.cu', 'sparse.cu', 'gemm.cu', 'umma.cu', 'umma_loss.cu', 'umma_score.cu', 'sampled.cu', 'mt_device.cu', 'optim.cu', 'dmf.cu', 'score.cu', 'dmf_topk.cu', 'host_rng.cpp', 'mt_jump.cpp']
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
         '-I', os.path.join(ROOT, 'include'), '-I', CSRC]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, 'include', 'drb.h'), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, 'build', src + '.o')
        cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-x', 'cu', '-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f'nvcc failed on {src}:\n{out}')
    link = [NVCC, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    subprocess.run(link, check=True)
    return LIB


if __name__ == '__main__':
    print(build_lib(force='--force' in sys.argv, verbose='-v' in sys.argv))
