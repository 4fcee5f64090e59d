"""CPU check of the warp FFT index maps: tools/host_check.cu runs the __host__ __device__ phase
functions of csrc/warp_fft.cuh lane by lane on the CPU and compares them with a direct DFT, for
both geometries of the group transform (PSFR_G_GEOM = 1 and 0).  Needs nvcc, no GPU."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    return None


@pytest.mark.parametrize('geom', [1, 0])
def test_host_check_fft_maps(tmp_path, geom):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip('nvcc not found')
    exe = str(tmp_path / ('host_check_g%d' % geom))
    subprocess.run([nvcc, '-O2', '-DPSFR_G_GEOM=%d' % geom, '-I', os.path.join(ROOT, 'muse_psfr_b200', 'csrc'),
                    os.path.join(ROOT, 'tools', 'host_check.cu'), '-o', exe], check=True, cwd=str(tmp_path))
    run = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, run.stdout + run.stderr
