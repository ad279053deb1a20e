"""Build libbpc_b200.so in-tree with nvcc for sm_100a (no GPU needed: nvcc cross-compiles).

    python -m bpc_baseline_b200.build [--force] [--verbose]

The shared library is a plain C-ABI object (include/bpc_b200.h); it does not link against torch.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libbpc_b200.so')
SOURCES = ['api.cu', 'match.cu', 'crop.cu', 'crop_cta.cu', 'gather.cu', 'jitter.cu']
HEADERS = ['common.cuh', 'geometry.cuh', 'lsap.cuh', 'crop_common.cuh']
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']


def nvcc_path() -> str:
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found (set NVCC=/path/to/nvcc)')


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(ROOT, 'include', 'bpc_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines=(), out: str = LIB) -> str:
    """``defines`` / ``out``: experiment builds (e.g. -DBPC_STG_CS into another file, selected with BPC_LIB).

    One object file per translation unit under build/obj (compiled in parallel, reused while the source, the headers and the
    defines are unchanged), then one link."""
    if not force and not stale() and out == LIB:
        return LIB
    import hashlib
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(ROOT, 'build', 'obj')
    os.makedirs(objdir, exist_ok=True)
    tag = hashlib.sha1(' '.join(sorted(defines)).encode()).hexdigest()[:8]
    base = [nvcc_path(), '-Xcompiler', '-fPIC', '-O3', '-std=c++17', '-lineinfo', '--fmad=false',
            *ARCH, '-I', os.path.join(ROOT, 'include'), '-I', CSRC]
    if verbose:
        base += ['-Xptxas', '-v']
    base += [f'-D{d}' for d in defines]
    hdrs = [os.path.join(CSRC, f) for f in HEADERS] + [os.path.join(ROOT, 'include', 'bpc_b200.h')]

    def compile_one(name):
        src = os.path.join(CSRC, name)
        obj = os.path.join(objdir, f'{os.path.splitext(name)[0]}-{tag}.o')
        newest = max(os.path.getmtime(d) for d in [src] + hdrs)
        if not force and not verbose and os.path.exists(obj) and os.path.getmtime(obj) > newest:
            return obj, None
        res = subprocess.run(base + ['-c', src, '-o', obj], capture_output=True, text=True)
        return obj, res

    with ThreadPoolExecutor(len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    for obj, res in results:
        if res is not None and (verbose or res.returncode != 0):
            sys.stderr.write(res.stdout + res.stderr)
        if res is not None and res.returncode != 0:
            raise RuntimeError(f'nvcc failed compiling {obj}')
    res = subprocess.run([nvcc_path(), '-shared', *ARCH, *[o for o, _ in results], '-o', out], capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError('nvcc failed linking libbpc_b200.so')
    return out


EXT = os.path.join(HERE, '_C.so')
EXT_SRC = os.path.join(CSRC, 'torch_ext.cpp')


def build_torch_ext(force: bool = False, verbose: bool = False) -> str:
    """bpc_baseline_b200/_C.so: the thin PyTorch C++ extension (csrc/torch_ext.cpp, torch.ops.bpc_b200.*) over the C ABI.

    Compiled in-tree with g++ against torch's headers and linked against libbpc_b200.so next to it (rpath $ORIGIN) --
    host code only, every kernel stays in libbpc_b200.so."""
    lib = build(force=force, verbose=verbose)
    deps = [EXT_SRC, os.path.join(ROOT, 'include', 'bpc_b200.h')]
    if not force and os.path.exists(EXT) and all(os.path.getmtime(d) <= os.path.getmtime(EXT) for d in deps):
        return EXT
    import torch
    from torch.utils import cpp_extension as ce
    cuda_home = os.path.dirname(os.path.dirname(nvcc_path()))
    inc = [p for p in ce.include_paths() if os.path.isdir(p)] + [os.path.join(cuda_home, 'include'), os.path.join(ROOT, 'include')]
    libdirs = [os.path.join(os.path.dirname(torch.__file__), 'lib'), os.path.join(cuda_home, 'lib64')]
    cmd = ['g++', '-shared', '-fPIC', '-O2', '-std=c++17', f'-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}',
           '-DTORCH_API_INCLUDE_EXTENSION_H', *[f'-I{p}' for p in inc], EXT_SRC, '-o', EXT,
           *[f'-L{d}' for d in libdirs], f'-L{HERE}', '-l:' + os.path.basename(lib),
           '-lc10', '-lc10_cuda', '-ltorch_cpu', '-ltorch_cuda', '-ltorch', '-lcudart',
           '-Wl,-rpath,$ORIGIN', *[f'-Wl,-rpath,{d}' for d in libdirs]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError('g++ failed building _C.so')
    return EXT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
    print(build_torch_ext(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
