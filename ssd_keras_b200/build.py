"""Build libssdk.so (sm_100a only) in-tree with nvcc.

``python -m ssd_keras_b200.build`` or ``build_library()``.  nvcc cross-compiles without a GPU.
The resulting ``ssd_keras_b200/_lib/libssdk.so`` is git-ignored but travels to the GPU box.
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIBDIR = os.path.join(HERE, '_lib')
LIB = os.path.join(LIBDIR, 'libssdk.so')

ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '-Xcompiler', '-ffp-contract=off',
          '-Xcudafe', '--diag_suppress=177', '-Xcudafe', '--diag_suppress=550']
# exactness-critical files: no FMA contraction on the device either
SOURCES = {
    'api.cu': ['--fmad=false'],
    'encode.cu': ['--fmad=false'],
    'decode.cu': ['--fmad=false'],
    'loss.cu': ['--fmad=false'],
    'batch.cu': ['--fmad=false'],
    'images.cu': ['--fmad=false'],
    'photometric.cu': ['--fmad=false'],
    'evaluate.cu': ['--fmad=false'],
    'conv.cu': [],
    'model.cu': [],
    'train.cu': [],
    'bn.cu': [],
    'wgrad.cu': [],
}


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', shutil.which('nvcc')):
        if c and os.path.exists(c):
            return c
    raise RuntimeError('nvcc not found')


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, '..', 'include')):
        for f in sorted(os.listdir(root)):
            if f.endswith(('.cu', '.cuh', '.h')):
                h.update(f.encode())
                h.update(open(os.path.join(root, f), 'rb').read())
    h.update(repr(SOURCES).encode())
    h.update(repr(COMMON).encode())
    return h.hexdigest()


def _compile(nvcc, src, extra, verbose):
    obj = os.path.join(LIBDIR, src.replace('.cu', '.o'))
    cmd = [nvcc] + ARCH + COMMON + extra + ['-c', os.path.join(CSRC, src), '-o', obj]
    if verbose:
        cmd.insert(1, '-Xptxas')
        cmd.insert(2, '-v')
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, obj, r


def build_library(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, 'build.stamp')
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    nvcc = _nvcc()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        for src, obj, r in ex.map(lambda s: _compile(nvcc, s, SOURCES[s], verbose), srcs):
            if verbose or r.returncode != 0:
                sys.stderr.write('== %s ==\n%s%s\n' % (src, r.stdout, r.stderr))
            if r.returncode != 0:
                raise RuntimeError('nvcc failed on %s' % src)
            objs.append(obj)
    cmd = [nvcc] + ARCH + ['-shared', '-o', LIB] + objs + ['-lcudart']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError('link failed')
    with open(stamp, 'w') as f:
        f.write(dig)
    return LIB


if __name__ == '__main__':
    print(build_library(force='--force' in sys.argv, verbose='-v' in sys.argv))
