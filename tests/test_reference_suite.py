"""Runs the reference's OWN single-process test files against this package (overlay package, see
tests/ref_suite/run.py).  290 reference tests; the multi-process files (partitioner, ddp, async_take, read_object …,
~12 min) are run with `python tests/ref_suite/run.py`.  Needs the reference's tests staged under oracle/_ref by build()
(oracle/make_ref.sh)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "tests")), reason="oracle/_ref/tests not staged (oracle/make_ref.sh)")
def test_reference_single_process_tests_pass_against_this_package():
    proc = subprocess.run(
        [sys.executable, os.path.join(ROOT, "tests", "ref_suite", "run.py"), "--fast"], capture_output=True, text=True, timeout=900
    )
    tail = "\n".join(proc.stdout.splitlines()[-15:])
    assert proc.returncode == 0, tail + proc.stderr[-2000:]
    assert " passed" in tail and " failed" not in tail, tail
