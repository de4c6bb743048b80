"""GPU: the kernel variants the environment knobs select -- the fp16 shortlist variants (PSB_TC16_EPI = 3 | 4,
PSB_TC16_MT = 2: csrc/catalog_tc.cu) and the 3xTF32 tcgen05 GEMM (csrc/gemm3_tf32.cu).  Each check runs in subprocesses under its own timeout (the knobs are
read once per process, and a hand-off bug in a tcgen05 pipeline hangs rather than fails); the bar is the one the
default kernels meet: the shortlist variants return the default kernel's ids and scores bit for bit, the GEMM is
within 5e-6 of an fp64 product."""
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


@pytest.mark.timeout(900)
def test_fp16_shortlist_variants_return_the_default_kernels_lists():
    out = _run("check_tc16_v2.py", "--quick", "--variants", "3,4,3/2,4/2", timeout=800)
    assert "every variant returns v1's lists bit for bit" in out


@pytest.mark.timeout(400)
def test_gemm3_tf32_matches_fp64_product():
    out = _run("check_gemm3.py", timeout=300)
    assert "within 5e-6" in out
