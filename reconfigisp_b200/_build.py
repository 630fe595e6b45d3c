"""In-tree build of the C-ABI shared library (nvcc, sm_100a only).

    python -m reconfigisp_b200._build [--force] [--verbose]

Every `csrc/*.cu` is compiled to `build/obj/*.o` (in parallel) and linked into
`reconfigisp_b200/libreconfigisp_b200.so`, which travels to the GPU box with the snapshot.
"""
import concurrent.futures as cf
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(ROOT, 'build', os.environ.get('RISP_BUILD_OBJ', 'obj'))
LIB = os.environ.get('RISP_BUILD_LIB', os.path.join(HERE, 'libreconfigisp_b200.so'))
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-O3', '-std=c++17', '-lineinfo', '-gencode', 'arch=compute_100a,code=sm_100a',
         '-Xcompiler', '-fPIC', '-Xptxas', '-v', '--expt-relaxed-constexpr'] + os.environ.get('RISP_BUILD_FLAGS', '').split()


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, '*.cu')))


def _digest(src):
    h = hashlib.sha1()
    for f in [src] + sorted(glob.glob(os.path.join(CSRC, '*.cuh'))) + [os.path.join(ROOT, 'include', 'reconfigisp_b200.h')]:
        with open(f, 'rb') as fh:
            h.update(fh.read())
    h.update(' '.join(FLAGS).encode())
    return h.hexdigest()


def _compile(src, force, verbose):
    obj = os.path.join(OBJ, os.path.basename(src)[:-3] + '.o')
    stamp = obj + '.sha1'
    dg = _digest(src)
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dg:
        return obj, ''
    cmd = [NVCC] + FLAGS + ['-c', src, '-o', obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('nvcc failed for %s:\n%s\n%s' % (src, r.stdout, r.stderr))
    with open(stamp, 'w') as fh:
        fh.write(dg)
    with open(obj + '.ptxas.log', 'w') as fh:
        fh.write(r.stderr)
    return obj, r.stderr if verbose else ''


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    srcs = _sources()
    with cf.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        res = list(ex.map(lambda s: _compile(s, force, verbose), srcs))
    objs = [o for o, _ in res]
    newest = max(os.path.getmtime(o) for o in objs)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [NVCC, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart']
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('link failed:\n%s\n%s' % (r.stdout, r.stderr))
    if verbose:
        for _, log in res:
            sys.stderr.write(log)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
