"""CPU: a model of the batched-affine rounds (msm_pair.cuh) built from the same pair templates the kernels run, compiled
with g++ (with and without the emulated PTX carry chains): sorted lists of real curve points with odd runs, runs across
thread boundaries, points at infinity, P + P over several rounds and P + (-P) keep every bucket sum on both curves."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("flags", [["-DSB_HOST_EMULATE_PTX"], []])
def test_host_batch_affine_rounds(tmp_path, flags):
    exe = str(tmp_path / "host_batch_affine_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", *flags, "-o", exe, os.path.join(ROOT, "tests", "host", "host_batch_affine_check.cpp")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "BATCH AFFINE CHECK PASSED" in out.stdout, out.stdout + out.stderr
