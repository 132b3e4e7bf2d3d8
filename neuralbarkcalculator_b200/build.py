"""Builds libnbc.so (all CUDA kernels + the C-ABI of include/nbc.h) in-tree with nvcc for sm_100a.

    python -m neuralbarkcalculator_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the repo snapshot."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libnbc.so')
SOURCES = ['api.cu', 'preprocess.cu', 'stem.cu', 'conv_tc.cu', 'conv_mma.cu', 'head.cu', 'ccl.cu', 'wce.cu', 'plan.cu',
           'train_kernels.cu', 'train_kernels2.cu', 'train_plan.cu', 'wgrad_tc.cu', 'lovasz.cu', 'eval.cu', 'augment.cu', 'png_host.cu', 'host_scan.cu']
FLAGS = ['-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-Xcompiler', '-fPIC',
         '--expt-relaxed-constexpr']


def _newest_source_mtime():
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'nbc.h')]
    return max(os.path.getmtime(p) for p in paths)


def needs_build():
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _newest_source_mtime()


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, 'build', src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [nvcc] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            failed = True
            sys.stderr.write('nvcc failed for %s:\n%s\n' % (src, out))
        elif verbose or out.strip():
            sys.stderr.write('[%s]\n%s\n' % (src, out))
    if failed:
        raise RuntimeError('libnbc.so build failed')
    subprocess.check_call([nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a'])
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
