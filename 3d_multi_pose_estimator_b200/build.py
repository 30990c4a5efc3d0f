"""Builds libb200pose.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m 3d_multi_pose_estimator_b200.build   (or: python 3d_multi_pose_estimator_b200/build.py)
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libb200pose.so')
SOURCES = ['common.cu', 'graph.cu', 'gat.cu', 'cluster.cu', 'lift.cu', 'gemm.cu', 'pack_json.cu', 'train.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return 'nvcc'


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'b200pose.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=True):
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, 'build', src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [_nvcc()] + NVCC_FLAGS + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError('nvcc failed on %s:\n%s' % (src, out.decode()))
        if verbose and out.strip():
            print(out.decode())
    cmd = [_nvcc(), '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    subprocess.check_call(cmd)
    if verbose:
        print('built', LIB)
    return LIB


if __name__ == '__main__':
    build(force='--force' in sys.argv)
