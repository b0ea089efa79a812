"""Build recipe for lib/libp3d.so: plain nvcc, sm_100a only, in-tree output (so it travels to the GPU box)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, 'csrc')
LIB = os.path.join(PKG, 'lib', 'libp3d.so')
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared']


def sources():
    return sorted(glob.glob(os.path.join(CSRC, '*.cu')))


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, '*.cuh')) + glob.glob(os.path.join(PKG, '..', 'include', '*.h'))
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(nvcc, src, obj, verbose):
    cmd = [nvcc] + [x for x in NVCC_FLAGS if x != '-shared'] + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return src, r.returncode, r.stdout


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into lib/libp3d.so (cross-compiles without a GPU).

    One object per translation unit under lib/obj/, compiled in parallel and only when stale (its own .cu, or any
    shared header, is newer), then one link step - so touching one kernel file costs one nvcc run, not seven."""
    if not force and not _stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        raise RuntimeError('nvcc not found: cannot build libp3d.so')
    objdir = os.path.join(os.path.dirname(LIB), 'obj')             # build products, git-ignored like the library itself
    os.makedirs(objdir, exist_ok=True)
    headers = glob.glob(os.path.join(CSRC, '*.cuh')) + glob.glob(os.path.join(PKG, '..', 'include', '*.h')) + [os.path.abspath(__file__)]
    t_hdr = max(os.path.getmtime(h) for h in headers)
    jobs, objs = [], []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + '.o')
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(t_hdr, os.path.getmtime(src)):
            jobs.append((src, obj))
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        results = list(ex.map(lambda j: _compile_one(nvcc, j[0], j[1], verbose), jobs))
    for src, rc, out in results:
        if rc != 0:
            sys.stderr.write(out)
            raise RuntimeError('nvcc failed on %s' % os.path.basename(src))
        if verbose:
            print(out)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)       # lib/ holds only ignored artefacts: a fresh clone has no such directory
    tmp = LIB + '.tmp.%d' % os.getpid()
    r = subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-o', tmp] + objs + ['-lz'],     # zlib: deflate + crc32 of the PNG writer (csrc/image_io.cu)
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError('nvcc failed linking libp3d.so')
    os.replace(tmp, LIB)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
