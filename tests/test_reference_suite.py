"""The reference's OWN host-logic tests, run unmodified against this package.

`anemoi-transform_b200/compat` serves `anemoi.transform.*` from anemoi_transform_b200, so the
reference's `tests/test_*.py` (matching, grouping, filter base classes, dispatching) import
this implementation instead of the reference's.  Runs only when ANEMOI_REFERENCE_SRC points at
the reference's sources (oracle/reference_import.py): its tests are not copied into this repo.
earthkit-data / anemoi-utils are not installed, so thin stand-ins (oracle/refstubs) provide the
few names the tests' fixtures need; tests that fetch data from the network skip themselves.
"""

import os
import re
import subprocess
import sys
from pathlib import Path

import pytest

from oracle import reference_import

REPO = Path(__file__).resolve().parent.parent
REF_TESTS = reference_import.REFERENCE_TESTS

pytestmark = [pytest.mark.reference, pytest.mark.skipif(REF_TESTS is None or not REF_TESTS.exists(), reason="reference tree not present")]

# host-logic test modules of the reference that exercise code on the hot path's host side
# (test_fields.py imports `src.anemoi.transform.fields` by path, i.e. the reference's own file, so it cannot be redirected)
MODULES = ["test_matching.py", "test_grouping.py", "test_filter.py", "test_dispatchingfilter.py", "test_create.py"]


def test_reference_host_tests_pass_against_this_package(tmp_path):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(
        [str(REPO / "anemoi-transform_b200" / "compat"), str(REPO / "anemoi-transform_b200"), str(REPO / "oracle" / "refstubs"), str(REPO)]
    )
    env.pop("ANEMOI_REFERENCE_SRC", None)
    cmd = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "--rootdir", str(REF_TESTS.parent), "-c", os.devnull, *[str(REF_TESTS / m) for m in MODULES]]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=tmp_path, timeout=600)
    tail = (r.stdout + r.stderr)[-3000:]
    m = re.search(r"(\d+) passed", r.stdout)
    assert "anemoi_transform_b200" in subprocess.run(
        [sys.executable, "-c", "import anemoi.transform.filter as f; print(f.SingleFieldFilter.__module__)"], capture_output=True, text=True, env=env
    ).stdout, "the shim did not resolve to this package"
    assert r.returncode == 0 and m, tail
    assert int(m.group(1)) >= 41, tail
