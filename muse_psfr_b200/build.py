"""Build libpsfr_b200.so in-tree with nvcc for sm_100a (no torch extension machinery).

    python -m muse_psfr_b200.build        # or: from muse_psfr_b200.build import build; build()

The shared library lands next to this file so that it travels with the repository
snapshot to the GPU box; it is git-ignored.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libpsfr_b200.so')
SOURCES = ['psfr_api.cu', 'psfr_passes.cu', 'psfr_hot.cu', 'psfr_hot2.cu', 'psfr_psd.cu', 'psfr_plane.cu', 'psfr_conv.cu',
           'psfr_energy.cu', 'psfr_ao.cu', 'psfr_band.cu']
HEADERS = ['psfr_internal.h', 'warp_fft.cuh', 'pass_kernel.cuh', 'fft_tables.h', 'fast_exp.cuh', 'tma.cuh', 'ee_geometry.h', '../../include/psfr.h']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden', '--expt-relaxed-constexpr']


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found: libpsfr_b200.so cannot be built (there is no CPU fallback)')


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the C-ABI shared library.
    Tuning experiments: PSFR_NVCC_EXTRA (environment) appends flags, e.g. -DPSFR_FIT_MINBLOCKS=3, and
    PSFR_LIB_TAG=x writes the variant to libpsfr_b200_x.so (loaded with PSFR_LIB_TAG=x as well)."""
    tag = os.environ.get('PSFR_LIB_TAG', '')
    lib = LIB if not tag else LIB.replace('.so', '_%s.so' % tag)
    if not force and not tag and not _stale():
        return LIB
    nvcc = _nvcc()
    extra = os.environ.get('PSFR_NVCC_EXTRA', '').split()
    objdir = os.path.join(HERE, 'build' + ('_' + tag if tag else ''))
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        cmd = [nvcc] + NVCC_FLAGS + extra + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError('nvcc failed on %s' % src)
        objs.append(obj)
    cmd = [nvcc, '-shared', '-o', lib] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    subprocess.check_call(cmd)
    return lib


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
