"""-m gpu: the persistent tcgen05 self-loop GEMM, run in a subprocess under a timeout so that a wrong descriptor can
only fail this test (the kernel traps instead of hanging), never poison the others."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_selfloop_gemm_matches_fp64_and_packed_kernel():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'selfloop_check.py')], capture_output=True, text=True,
                       timeout=300)
    sys.stdout.write(r.stdout)
    sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0 and 'SELFLOOP_OK' in r.stdout
