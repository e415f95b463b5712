"""Builds libcgg_b200.so (the C-ABI library, include/cgg_b200.h) in-tree with nvcc for
sm_100a.  `python -m cgg_b200.build` or __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libcgg_b200.so')
SOURCES = ['kernels_f32.cu', 'train_kernels.cu', 'post_kernels.cu', 'match_kernels.cu', 'caption_kernels.cu', 'pixdec_kernels.cu', 'gemm_tc.cu', 'gemm_tf32.cu', 'attention_tc.cu', 'path_bf16.cu', 'api.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC']


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def needs_build():
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(os.path.dirname(HERE), 'include', 'cgg_b200.h')]
    return (not os.path.exists(LIB)) or os.path.getmtime(LIB) < _newest(deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace('.cu', '.o'))
        extra = os.environ.get('CGG_NVCC_EXTRA', '').split()      # extra nvcc flags, e.g. -Xptxas -warn-spills
        cmd = [nvcc] + NVCC_FLAGS + extra + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError('nvcc failed on %s' % src)
    cmd = [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-o', LIB] + objs + ['-lcuda']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError('link failed')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
