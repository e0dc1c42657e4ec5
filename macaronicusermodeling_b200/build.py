"""Build libmlbp.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libmlbp.so')
STAMP = os.path.join(HERE, 'libmlbp.so.stamp')
SOURCES = ['api.cu', 'tables.cu', 'unary.cu', 'messages.cu', 'gemm_simt.cu', 'gemm_tcgen05.cu', 'gradient.cu',
           'dense.cu', 'rescore.cu', 'spikes.cu', 'topk.cu', 'format.cu', 'parse.cu', 'joint.cu', 'maxprod.cu',
           'plan.cpp']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '--use_fast_math=false',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=default']


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), 'include')):
        for name in sorted(os.listdir(root)):
            if name.endswith(('.cu', '.cuh', '.cpp', '.h')):
                with open(os.path.join(root, name), 'rb') as f:
                    h.update(name.encode())
                    h.update(f.read())
    h.update((' '.join(NVCC_FLAGS) + os.environ.get('MLBP_EXTRA_NVCC_FLAGS', '')).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every CUDA / C++ source of the package into macaronicusermodeling_b200/libmlbp.so."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    flags = [f for f in NVCC_FLAGS if f != '--use_fast_math=false'] + os.environ.get('MLBP_EXTRA_NVCC_FLAGS', '').split()
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, 'build', src.rsplit('.', 1)[0] + '.o')
        cmd = [nvcc] + flags + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write('---- %s\n%s\n' % (src, out))
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed building libmlbp.so')
    subprocess.check_call([nvcc, '-shared', '-o', LIB] + objs + ['-lcudart'])
    with open(STAMP, 'w') as f:
        f.write(dig)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
