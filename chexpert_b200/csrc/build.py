"""Build libaaconv_b200.so in-tree with nvcc for sm_100a (no torch headers, no libcuda link).

    python chexpert_b200/csrc/build.py [--force]

The shared object is git-ignored but travels with the gpurun snapshot.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ['api.cu', 'runtime.cu', 'prologue.cu', 'bn_relu.cu', 'bn_cl.cu', 'fp32_gemms.cu', 'fp32_attn.cu', 'fp32_path.cu', 'bce.cu', 'eval_ops.cu', 'bf16_path.cu', 'tc_host.cu', 'aug_ops.cu', 'aug_tc.cu', 'attn_tc.cu', 'attn_cc.cu', 'attn_tc_bwd.cu', 'gemm_tc.cu', 'prep.cu', 'cam.cu']
LIB = os.path.join(HERE, 'libaaconv_b200.so')
BUILD_DIR = os.path.join(HERE, 'build')
NVCC = '/usr/local/cuda/bin/nvcc'
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def _digest():
    h = hashlib.sha256()
    for root, _, files in os.walk(HERE):
        for f in sorted(files):
            if f.endswith(('.cu', '.cuh', '.h', '.py')):
                h.update(open(os.path.join(root, f), 'rb').read())
    h.update(open(os.path.join(HERE, '..', '..', 'include', 'aaconv_b200.h'), 'rb').read())
    return h.hexdigest()


def build(force=False, verbose=True):
    stamp = os.path.join(BUILD_DIR, 'stamp')
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    os.makedirs(BUILD_DIR, exist_ok=True)

    def cc(src):
        obj = os.path.join(BUILD_DIR, src.replace('.cu', '.o'))
        cmd = [NVCC, *FLAGS, '-c', os.path.join(HERE, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(BUILD_DIR, src + '.log')
        open(log, 'w').write(r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError(f'nvcc failed for {src}:\n{r.stdout}\n{r.stderr}')
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(cc, SOURCES))
    cmd = [NVCC, '-shared', '-o', LIB, *objs, '-gencode', 'arch=compute_100a,code=sm_100a', '-cudart', 'static']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    open(stamp, 'w').write(dig)
    if verbose:
        print('built', LIB)
    return LIB


if __name__ == '__main__':
    build(force='--force' in sys.argv)
