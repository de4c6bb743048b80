"""GPU: the 3xTF32 tcgen05 GEMM (csrc/gemm3_tf32.cu) on its own, within 5e-6 of an fp64 product.  The check runs in a
subprocess under its own timeout (a hand-off bug in a tcgen05 pipeline hangs rather than fails)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _run(script, *args, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", script)] + list(args), capture_output=True,
                       text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-500:])
    return r.stdout


@pytest.mark.timeout(400)
def test_gemm3_tf32_matches_fp64_product():
    out = _run("check_gemm3.py", timeout=300)
    assert "within 5e-6" in out
