"""Build libnbasr.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc. No torch dependency."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(CSRC, 'libnbasr.so')
SOURCES = ['api.cu', 'tma_maps.cu', 'gemm_simt.cu', 'gemm2_sm100.cu', 'elementwise.cu', 'layernorm2.cu', 'gconv.cu', 'gconv_sm100.cu', 'lstm.cu', 'lstm_sm100.cu', 'sequence.cu', 'ctc_align.cu', 'edit_align.cu', 'optim.cu', 'gate_gram.cu', 'pack_batch.cu', 'frontend.cu']
NVCC_FLAGS = ['-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr', '-Xptxas', '-v']


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return 'nvcc'


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh', '.h'))]
    deps.append(os.path.join(os.path.dirname(HERE), 'include', 'nbasr.h'))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []

    def compile_one(src):
        obj = os.path.join(CSRC, src.replace('.cu', '.o'))
        cmd = [nvcc] + NVCC_FLAGS + ['-c', os.path.join(CSRC, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed for {src}:\n{r.stdout}\n{r.stderr}')
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
