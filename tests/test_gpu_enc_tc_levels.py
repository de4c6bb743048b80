"""GPU: the encoder's tensor-core path (the default) against the fp32 FFMA kernels (PSB_ENC_TC=0), stage by stage.

The knob is read once per process, so each path runs in a subprocess of its own (profiles/diff_enc_tc.py for the
forward pass's saved activations, profiles/diff_enc_bwd_tc.py for every gradient of the backward pass): the default
path (projections and both tails on tcgen05) and the FFMA path both stay runnable and in agreement -- within 2e-5 of
each tensor's maximum in the scripts, measured 1.3e-6 / 2.2e-6 (DESIGN.md section 4)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(script):
    env = {k: v for k, v in os.environ.items() if k != "PSB_ENC_TC"}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", script)], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout


def test_forward_levels_agree_with_the_ffma_kernels():
    out = _run("diff_enc_tc.py")
    assert "agree with the FFMA kernels stage by stage" in out


def test_backward_levels_agree_with_the_ffma_kernels():
    out = _run("diff_enc_bwd_tc.py")
    assert "tensor-core backward agrees with the FFMA kernels" in out
