"""Builds libv2v_b200.so (sm_100a) in-tree with nvcc.  No GPU is needed to build."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
SOURCES = ['conv_umma.cu', 'conv_simt.cu', 'norm.cu', 'layout.cu', 'warp.cu', 'pyramid.cu', 'flowops.cu', 'flownet_glue.cu', 'backward.cu', 'wgrad_umma.cu', 'losses.cu', 'face.cu', 'plan.cu',
           'api.cu']
LIB = os.path.join(HERE, 'libv2v_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
         '--expt-relaxed-constexpr', '-cudart', 'static']


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'v2v_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    procs = []
    for s in SOURCES:
        o = os.path.join(HERE, 'build', s.replace('.cu', '.o'))
        cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, s), '-o', o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write('---- %s\n%s\n' % (s, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed')
    cmd = [NVCC, '-shared', '-o', LIB] + objs + ['-cudart', 'static', '-gencode', 'arch=compute_100a,code=sm_100a']
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
