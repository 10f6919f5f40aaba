"""Builds libmoog_b200.so (the sm_100a kernels + C ABI) in-tree with nvcc.

    python -m moog_b200.build          # or: moog_b200.build.build()

The library is plain CUDA C++ behind an `extern "C"` boundary
(include/moog_b200.h); it does not link against torch.  `-fmad=false` is part
of the numerical contract: the kernels follow the reference's float64 /
float32 operation order and only fuse where the reference's BLAS does.
"""
import os
import subprocess
import sys

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, 'csrc')
LIB = os.environ.get('MOOG_B200_LIB') or os.path.join(_PKG, 'lib', 'libmoog_b200.so')   # override: A/B runs
SOURCES = ['moog_step.cu', 'moog_render.cu', 'moog_observe.cu', 'moog_rays.cu', 'moog_capi.cu', 'moog_host_geom.cpp']
HEADERS = [os.path.join(CSRC, 'moog_common.cuh'), os.path.join(CSRC, 'moog_render_dev.cuh'),
           os.path.join(CSRC, 'moog_dcv_argmin.cuh'), os.path.join(CSRC, 'moog_seg_cross.cuh'),
           os.path.join(_PKG, '..', 'include', 'moog_b200.h'),
           os.path.join(_PKG, '..', 'include', 'moog_b200_program.h')]

# MOOG_NVCC_OPT: optimisation flags of an experimental build (A/B runs together with MOOG_B200_LIB)
NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo'] + os.environ.get('MOOG_NVCC_OPT', '-O3').split() + [
    '-std=c++17', '-fmad=false', '-prec-div=true', '-prec-sqrt=true',
    '--expt-extended-lambda', '-Xcompiler', '-fPIC,-ffp-contract=off',
    '-Wno-deprecated-gpu-targets',
] + (['-DMOOG_PROFILE_PHASES'] if os.environ.get('MOOG_PROFILE_PHASES') else []) + (
    ['-DMOOG_PROFILE_DCV'] if os.environ.get('MOOG_PROFILE_DCV') else []) + (
    ['-DMOOG_PROFILE_GCV'] if os.environ.get('MOOG_PROFILE_GCV') else []) + (
    ['-DMOOG_PROFILE_INTEG'] if os.environ.get('MOOG_PROFILE_INTEG') else [])


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return 'nvcc'


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile when sources are newer than the library; returns its path."""
    if not (force or is_stale()):
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(_PKG, 'lib', os.path.splitext(src)[0] + '.o')
        cmd = [_nvcc()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + [
            '-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((cmd, subprocess.Popen(cmd)))
        objs.append(obj)
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError('nvcc failed: ' + ' '.join(cmd))
    # (the arch again at the link step: without it nvcc adds an empty default-arch device stub to the library)
    cmd = [_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs + ['-lcudart']
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
