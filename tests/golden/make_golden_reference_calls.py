#!/usr/bin/env python
"""Writes tests/golden/reference_calls.json: runs the tests that call the reference's compiled code (oracle/_ref,
built by oracle/build_ref.py and oracle/build_ref_cxx.py from a simpledet checkout) with SDET_RECORD_REFERENCE=1,
which records a digest of every result next to the arguments of the call (tests/reference_replay.py).

Run:  python tests/golden/make_golden_reference_calls.py     (needs the compiled reference)"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TESTS = ["tests/test_oracle_ref_cxx.py", "tests/test_oracle_ref.py::test_live_against_compiled_reference"]

if __name__ == "__main__":
    out = os.path.join(HERE, "reference_calls.json")
    if os.path.exists(out):
        os.remove(out)  # a fresh recording: no entries of tests that no longer exist
    sys.exit(subprocess.call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *TESTS], cwd=ROOT,
                             env=dict(os.environ, SDET_RECORD_REFERENCE="1")))
