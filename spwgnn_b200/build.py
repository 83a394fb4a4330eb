"""Compile spwgnn_b200/csrc/spwgnn.cu into spwgnn_b200/libspwgnn.so for sm_100a (in-tree)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'csrc', 'spwgnn.cu')
DEPS = [os.path.join(HERE, 'csrc', f) for f in ('spwgnn.cu', 'spw_common.cuh', 'spw_edges.cuh', 'spw_kernels.cuh', 'spw_tc.cuh', 'spw_rows_tc.cuh', 'spw_pipe_tc.cuh', 'spw_csl.cuh', 'spw_csl_kernels.cuh', 'spw_csl_wgrad.cuh', 'spw_csl_path.inl', 'spw_small.cuh', 'spw_small_grad.cuh', 'spw_obj_grad.cuh', 'spw_rel_grad.cuh', 'spw_input_grad.cuh')] + \
       [os.path.join(os.path.dirname(HERE), 'include', 'spwgnn.h')]
OUT = os.path.join(HERE, 'libspwgnn.so')
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '--shared',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=default']


def find_nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found')


def build(force=False, verbose=False):
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    cmd = [find_nvcc()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', OUT, SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return OUT


if __name__ == '__main__':
    print(build(force=True, verbose=True))
