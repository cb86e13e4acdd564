"""The trunk kernels launched in plain stream order (SPECB200_PDL=0) instead of with programmatic dependent launch: the
conv-kernel and whole-path 16-bit parity tests, run in a subprocess with the switch set (it is read once per process).  This
is the baseline for ruling out an ordering bug in the programmatic edges.  It only runs when SPECB200_RUN_EXPERIMENTAL=1, so
that a routine GPU run spends its time on the default path:

    SPECB200_RUN_EXPERIMENTAL=1 python -m pytest tests/test_gpu_experimental.py -m gpu -q"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get('SPECB200_RUN_EXPERIMENTAL') != '1', reason='set SPECB200_RUN_EXPERIMENTAL=1 to run the non-default launch mode')
@pytest.mark.parametrize('switch,value', [('SPECB200_PDL', '0')])
def test_non_default_variant_keeps_parity(switch, value):
    env = dict(os.environ)
    env[switch] = value
    r = subprocess.run([sys.executable, '-m', 'pytest', os.path.join(ROOT, 'tests', 'test_gpu_parity.py'), '-m', 'gpu', '-x', '-q',
                        '-k', 'conv_kernels or full_forward_lowp_parity or golden or ragged'],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
