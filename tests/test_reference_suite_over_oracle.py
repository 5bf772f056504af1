"""The reference's own code, byte-compiled by ``build()`` into oracle/_ref (oracle/ref_build.py);
skipped where no build has staged it:

* the reference's own test files run, unmodified, over its own Pink-layer code with the oracle
  standing in for the third-party primitives (scripts/run_reference_tests.py; committed record:
  profiles/r02j_reference_tests_over_oracle.txt) - no failure other than the three that assert
  the geometry of a robot that is not available offline;
* the same files against THIS package (module name ``pink`` bound to ``pink_b200``, engine = host
  build of the kernels; record profiles/r02k_reference_tests_on_product_host_build.txt);
* re-running the reference reproduces the committed ``tests/golden/ref_pink_layer_*.npz``."""

import os
import re
import subprocess
import sys

import pytest

from oracle import ref_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not ref_build.staged(), reason="no reference staged in oracle/_ref by build()")


@needs_reference
def test_reference_test_suite_passes_over_the_oracle(tmp_path):
    record = tmp_path / "record.txt"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "run_reference_tests.py"), str(record)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    text = record.read_text()
    assert "# unexpected failures: 0" in text
    passed = int(re.search(r"(\d+) passed", text).group(1))
    assert passed >= 110, text[:400]
    # the finite-difference Jacobian tests of the reference are among them
    assert re.search(r"^PASSED\s+test_jacobians.py::TestJacobians::test_frame_task", text, re.M)


@needs_reference
def test_reference_test_suite_against_this_package_on_the_host_build(tmp_path):
    """``pink`` -> ``pink_b200`` (tests/refalias_plugin.py), engine = host build of the kernels: the
    reference's own tests as the drop-in check of the Python mirror.  Failures are allowed only where
    the runner names the cause (robots that are not available offline, fp64 tolerances on an fp32
    engine, Pinocchio's ``data.J``)."""
    record = tmp_path / "record.txt"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "run_reference_tests.py"), "--product", str(record)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    text = record.read_text()
    assert "# unexpected failures: 0" in text
    assert int(re.search(r"(\d+) passed", text).group(1)) >= 100, text[:400]


@needs_reference
def test_reference_run_reproduces_the_committed_pink_layer_fixtures():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "make_reference_golden.py"), "--check"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    from tests import ref_pink_layer_cases

    assert res.stdout.count("committed fixture reproduced") == len(ref_pink_layer_cases.NAMES) + len(ref_pink_layer_cases.EXAMPLE_LOOPS)
