"""
Build the two in-tree libraries:
  libbin3c_b200.so  the device path, nvcc for sm_100a (cross-compiles without a GPU)
  libbin3c_io.so    the host-side BAM pair reader and edge-list writer, g++ + zlib + pthreads
    python -m bin3c_b200.csrc.build [--force] [-v]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, 'libbin3c_b200.so')
SOURCES = ['core.cu', 'accum.cu', 'rowops.cu', 'kr.cu', 'synth.cu', 'bamdec.cu', 'sites.cu', 'edgefmt.cu', 'bgzf.cu']
HEADERS = ['common.cuh', 'inflate.cuh', 'deflate.cuh', 'bgzf.cuh', 'sites.cuh', 'edgefmt.cuh', 'edgefmt_pow5.h', os.path.join('..', '..', 'include', 'bin3c_b200.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '--shared']


IO_LIB = os.path.join(PKG, 'libbin3c_io.so')
IO_SOURCES = ['io_bam.cpp', 'io_edges.cpp']
IO_HEADERS = ['io_common.h', os.path.join('..', '..', 'include', 'bin3c_io.h')]
IO_FLAGS = ['-O2', '-std=c++17', '-Wall', '-fPIC', '-shared', '-pthread']


def build_io(force=False):
    deps = [os.path.join(HERE, f) for f in IO_SOURCES + IO_HEADERS] + [os.path.abspath(__file__)]
    if not force and os.path.exists(IO_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(IO_LIB) for d in deps):
        return IO_LIB
    cmd = [os.environ.get('CXX', 'g++')] + IO_FLAGS + [os.path.join(HERE, f) for f in IO_SOURCES] + ['-o', IO_LIB, '-lz']
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError('g++ failed:\n' + res.stdout)
    return IO_LIB


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError('nvcc not found')


OBJ_DIR = os.path.join(HERE, '_build')


def _deps_common():
    return [os.path.join(HERE, f) for f in HEADERS] + [os.path.abspath(__file__)]


def _obj(src):
    return os.path.join(OBJ_DIR, os.path.splitext(src)[0] + '.o')


def _obj_stale(src):
    o = _obj(src)
    if not os.path.exists(o):
        return True
    t = os.path.getmtime(o)
    return any(os.path.getmtime(d) > t for d in [os.path.join(HERE, src)] + _deps_common())


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, f) for f in SOURCES] + _deps_common()
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, only when stale), then one link."""
    build_io(force)
    if not force and not stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != '--shared']

    def compile_one(src):
        if not force and not _obj_stale(src):
            return ''
        cmd = [_nvcc()] + flags + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(HERE, src), '-o', _obj(src)]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            raise RuntimeError('nvcc failed on {}:\n{}'.format(src, res.stdout))
        return res.stdout

    with ThreadPoolExecutor(len(SOURCES)) as ex:
        logs = list(ex.map(compile_one, SOURCES))
    cmd = [_nvcc(), '--shared', '-Xcompiler', '-fPIC', '-gencode', 'arch=compute_100a,code=sm_100a'] + \
          [_obj(f) for f in SOURCES] + ['-o', LIB]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc link failed:\n' + res.stdout)
    if verbose:
        print('\n'.join(logs))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
