"""The CUDA kernel SOURCE, compiled for the host by tools/emu (warps as fibers, shuffles / async copies emulated; test
tooling like oracle/, never loaded by the package) and checked against the oracle: lets the GPU-less `-m "not gpu"` run
exercise the kernels' logic -- op-list compiler, table stream and ring, dynamic group schedule, sorted-keeps fork, staging
pipeline, multi-device dealing -- bit for bit.  The GPU tests remain the parity proof."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")


@pytest.fixture(scope="module")
def emu_built():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def _check(flt):
    r = subprocess.run([sys.executable, os.path.join(EMU, "check.py"), flt], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-3000:] + r.stderr[-2000:]
    assert "mismatching=   0" in r.stdout
    return r.stdout


def test_every_kernel_family_matches_the_oracle_under_the_emulator(emu_built):
    out = _check("")
    assert out.count("kernel=scl_lut_warp") >= 15 and "kernel=path_warp" in out

