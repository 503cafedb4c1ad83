"""Drop-in check: the cases of the REFERENCE'S OWN test suite that need no device, restated in tests/reference_cases.py,
run against this package through compat/ (a `tensorrec` alias package, a torch-backed `tensorflow` stand-in for the
handful of TF names those tests use, and a `nose_parameterized` shim) in a process of their own.  Every case the
reference's unmodified test files passed with (tests/golden/reference_suite_cases.json) must pass.  The reference tests
that reach predict / predict_rank need a CUDA device (no CPU fallback) and are restated by this repo's own GPU tests
(tests/test_api_gpu.py, tests/test_kernels_gpu.py)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'reference_suite_cases.json')))
TARGETS = [t for t in GOLDEN if not t.startswith('_')]


@pytest.mark.parametrize('target', TARGETS, ids=[t.replace('::', '-') for t in TARGETS])
def test_reference_cases_pass_through_compat(tmp_path, target):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, 'compat'), ROOT]), CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, '-m', 'tests.reference_cases', target], capture_output=True, text=True,
                         timeout=900, cwd=str(tmp_path), env=env)
    tail = out.stdout[-3000:] + out.stderr[-3000:]
    passed = sorted(line.split(' ', 1)[1] for line in out.stdout.splitlines() if line.startswith('PASS '))
    assert out.returncode == 0 and passed == GOLDEN[target], tail
