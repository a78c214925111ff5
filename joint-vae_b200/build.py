"""Builds libjvae_sm100.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting .so travels to
the GPU box with the repo snapshot.  Usage:  python joint-vae_b200/build.py [--force] [--verbose]
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libjvae_sm100.so')
STAMP = os.path.join(HERE, 'build', 'stamp.txt')

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC']


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _digest():
    h = hashlib.sha256()
    files = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h')))
    files.append(os.path.join(HERE, '..', 'include', 'jvae_b200.h'))
    for f in files:
        with open(f, 'rb') as fh:
            h.update(os.path.basename(f).encode())      # not the absolute path: the tree moves between machines
            h.update(fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def current():
    """Whether the library was built from the present sources and flags (reads only)."""
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _digest()


def build(force=False, verbose=False):
    """Compiles csrc/*.cu when the sources changed since the last build.  Safe to call from several processes at once
    (one rank per GPU under torchrun): an exclusive file lock serialises them and the late comers find the fresh stamp."""
    import fcntl
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    with open(os.path.join(HERE, 'build', '.lock'), 'w') as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force, verbose):
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    dig = _digest()
    if not force and current():
        return LIB
    if not os.path.exists(nvcc):
        if os.path.exists(LIB):      # GPU box without toolkit changes: use the prebuilt library
            return LIB
        raise RuntimeError(f'nvcc not found at {nvcc} and {LIB} is not built')
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(HERE, 'build', os.path.basename(src)[:-3] + '.o')
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f'--- {os.path.basename(src)}\n{out}\n')
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError('nvcc failed')
    # static cudart (nvcc default): the library shares the primary context with PyTorch; the driver API
    # (cuTensorMapEncodeTiled) is resolved at run time through cudaGetDriverEntryPoint, so no -lcuda
    cmd = [nvcc, '-shared', '-o', LIB] + objs
    subprocess.run(cmd, check=True)
    with open(STAMP, 'w') as f:
        f.write(dig)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
