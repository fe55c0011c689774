"""Build libvlnimagine.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libvlnimagine.so')
SOURCES = ['vi_api.cu', 'vi_gemm_tc.cu', 'vi_gemm_simt.cu', 'vi_attn.cu', 'vi_rows.cu', 'vi_bwd.cu', 'vi_wgrad.cu', 'vi_attn_bwd.cu', 'vi_graph.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared', '-lcudart']


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'vlnimagine.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for src in SOURCES:                      # compile units in parallel, then link
        obj = os.path.join(HERE, 'build', src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [nvcc, '-c', os.path.join(CSRC, src), '-o', obj] + [f for f in NVCC_FLAGS if f not in ('-shared', '-lcudart')]
        if verbose:
            cmd += ['-Xptxas', '-v']
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write('--- %s ---\n%s\n' % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed building libvlnimagine.so')
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart']
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
