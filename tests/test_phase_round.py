"""csrc/phase_round.cuh on the CPU: the fused phase kernel's FMA-pipe rounding of the DM phase to int32 fixed point."""
import os
import shutil
import subprocess

import pytest


def test_phase_fixed_rn_is_float2int_rn_for_every_input(tmp_path):
    """phase_fixed_rn(d) == round-to-nearest-even(d * 2^22), which is __float2int_rn(d * 2^22), for each of the
    2,281,701,376 floats with |d| < 512: every input the conversion does not saturate."""
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not found')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / 'phase_round_host')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-Xcompiler', '-fopenmp', '-Wno-deprecated-gpu-targets', '-o', exe,
                    os.path.join(root, 'tools', 'micro', 'phase_round_host.cu')], check=True, capture_output=True)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    bad, n = map(int, out.stdout.split())
    assert n == 2 * 0x44000000 and bad == 0 and out.returncode == 0, out.stdout
