"""Build libmonoloco_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Every .cu is compiled to an object in parallel (only the stale ones), then linked into one shared library."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_DIR = os.path.join(HERE, 'lib')
OBJ_DIR = os.path.join(LIB_DIR, 'obj')
LIB_PATH = os.path.join(LIB_DIR, 'libmonoloco_b200.so')
HEADER = os.path.join(HERE, '..', 'include', 'monoloco_b200.h')
SOURCES = ['model.cu', 'forward.cu', 'forward_small.cu', 'forward_wide.cu', 'forward_wide2.cu', 'train.cu', 'optim.cu', 'post.cu', 'probe_tc.cu', 'forward_tc.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC']


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))] + [HEADER]


def _obj(src):
    return os.path.join(OBJ_DIR, os.path.splitext(src)[0] + '.o')


def _stale_objects(force):
    hdr_t = max(os.path.getmtime(h) for h in _headers())
    out = []
    for s in SOURCES:
        o, c = _obj(s), os.path.join(CSRC, s)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(c), hdr_t):
            out.append(s)
    return out


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    stale = _stale_objects(force)
    if not stale and os.path.exists(LIB_PATH) and \
            os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(_obj(s)) for s in SOURCES):
        return LIB_PATH

    def compile_one(s):
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, s), '-o', _obj(s)]
        return s, subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(stale)))) as ex:
        results = list(ex.map(compile_one, stale))
    failed = False
    for s, res in results:
        if verbose or res.returncode != 0:
            sys.stderr.write("---- %s\n%s" % (s, res.stdout))
        failed |= res.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed building libmonoloco_b200.so')
    link = [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-o', LIB_PATH] + [_obj(s) for s in SOURCES]
    res = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise RuntimeError('nvcc failed linking libmonoloco_b200.so')
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
