"""CPU, only where PMMH_REFERENCE_ROOT points at a checkout of the reference (compops/pmmh-qn) and
oracle/build_ref.py has built its kernels: the reference's unmodified quasi-Newton sampler and Cython
estimator run under the lock-step front-end (parameter/lockstep.py).  The sampler is the reference's own
Python code, which this project does not carry, so the test cannot run without that checkout.
The check itself runs in a subprocess: importing the reference changes global interpreter state."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_ROOT = os.environ.get("PMMH_REFERENCE_ROOT")


@pytest.mark.skipif(not (REF_ROOT and os.path.isdir(os.path.join(REF_ROOT, "python"))),
                    reason="needs PMMH_REFERENCE_ROOT set to a checkout of the reference")
def test_reference_sampler_under_the_lockstep_front_end():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "lockstep_reference_check.py")],
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    out = json.loads(proc.stdout.strip().splitlines()[-1])
    assert out["single_chain_equals_recorded_run"], out
    assert out["three_chains_lockstep_equal_solo"], out
    assert out["batch_sizes"] and max(out["batch_sizes"]) == 3, out
