"""Build libxna_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m xna_basecaller_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libxna_b200.so')
SOURCES = ["xb_api.cu", "crf_decode.cu", "crf_decode_lin.cu", 'conv_stem.cu', 'gemm_tc.cu', 'conv3_gemm.cu', 'lstm_persistent.cu', 'inproj_gemm.cu', 'misc_kernels.cu', 'preprocess.cu', 'train_bwd.cu', 'lstm_bptt.cu', 'wgrad_gemm.cu', 'optim.cu', 'beam_search.cu', 'align.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-cudart', 'static']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu into an object (only the stale ones) and link the shared library."""
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    headers.append(os.path.join(HERE, '..', 'include', 'xna_basecaller.h'))
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    objs, procs = [], []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        objs.append(obj)
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + NVCC_FLAGS + ['-c', path, '-o', obj]
            if verbose:
                print(' '.join(cmd))
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError('nvcc failed on %s:\n%s' % (src, out.decode()))
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-cudart', 'static', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs
        subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
