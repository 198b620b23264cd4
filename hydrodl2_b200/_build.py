"""Build the C-ABI CUDA library in-tree with nvcc for sm_100a.

    python -m hydrodl2_b200._build [--force] [--verbose]

Output: ``hydrodl2_b200/lib/libhbv_b200.so`` (git-ignored, shipped to the GPU
box by gpurun).  cudart is linked statically so the library is self-contained
and can be loaded from C, ctypes or next to PyTorch's own runtime (both use the
device's primary context, so PyTorch device pointers and streams are valid).
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIBDIR = os.path.join(HERE, 'lib')
LIB = os.path.join(LIBDIR, 'libhbv_b200.so')
SOURCES = ['hbv_cabi.cu', 'hbv_fwd.cu', 'hbv_bwd.cu', 'uh_route.cu', 'pair_route.cu', 'hbv_adj.cu',
           'hbv_dense.cu', 'hbv_lean.cu', 'hbv_pipe.cu', 'fill.cu', 'allreduce.cu', 'hbv_tlm.cu']
HEADERS = ['hbv_step.cuh', 'hbv_common.cuh', 'hbv_tlm.cuh', os.path.join('..', '..', 'include', 'hbv_b200.h')]
# Translation units whose explicit template instantiations are compiled as several objects in
# parallel (-DHBV_TU_PART=k; the source emits all of them when the macro is absent): the
# standard-layout and the stage-pipelined kernels are a few hundred instantiations each and would
# otherwise be the critical path of the build.
PARTS = {'hbv_lean.cu': 4, 'hbv_pipe.cu': 2}

NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a',
    '-O3', '-lineinfo', '-std=c++17',
    '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden',
    '--expt-relaxed-constexpr',
]


def nvcc_path() -> str:
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found: the CUDA library cannot be built')


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, math: int | None = None) -> str:
    """Compile every .cu for sm_100a and link the shared library.  Returns its path.

    math=0 builds the precise-math variant (IEEE division, libdevice powf/expf/logf) as
    ``lib/libhbv_b200_precise.so``; the default library uses the SFU path (hbv_step.cuh)."""
    out = LIB if math is None else os.path.join(LIBDIR, 'libhbv_b200_precise.so' if math == 0
                                                else f'libhbv_b200_math{math}.so')
    if math is None and not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = nvcc_path()
    objs = []
    procs = []
    tag = '' if math is None else f'_m{math}'
    extra = [] if math is None else [f'-DHBV_MATH={math}']
    units = []          # (source, object suffix, extra defines); the many-instantiation units first
    for s in sorted(SOURCES, key=lambda n: -PARTS.get(n, 1)):
        n = PARTS.get(s, 1)
        units += [(s, '', [])] if n == 1 else [(s, f'_p{k}', [f'-DHBV_TU_PART={k}']) for k in range(1, n + 1)]
    for s, suffix, defs in units:
        o = os.path.join(LIBDIR, s.replace('.cu', f'{suffix}{tag}.o'))
        cmd = [nvcc, *NVCC_FLAGS, *extra, *defs, '-c', os.path.join(CSRC, s), '-o', o]
        if verbose:
            cmd.insert(1, '-Xptxas')
            cmd.insert(2, '-v')
            print(' '.join(cmd))
        procs.append((s + suffix, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s, p in procs:
        log, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f'nvcc failed on {s}:\n{log}')
        if verbose and log:
            print(log)
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', out, *objs]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'link failed:\n{r.stdout}')
    return out


if __name__ == '__main__':
    path = build(force='--force' in sys.argv, verbose='--verbose' in sys.argv,
                 math=0 if '--precise' in sys.argv else None)
    print(path)
