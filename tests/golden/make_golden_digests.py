"""Regenerates tests/golden/reference_digests.json: the digests (tests/common.py:digest) of what the UNMODIFIED
reference library oracle/_ref/libnrsc5_ref.so answers in the tests that call tests/common.py:assert_reference.  It
runs those tests with NRSC5_WRITE_REF_DIGESTS=1, which makes assert_reference record the reference's answer before
it checks the restatement against it.  Needs the reference library; the JSON is committed.

    python tests/golden/make_golden_digests.py
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TESTS = ["tests/test_oracle.py", "tests/test_oracle_am.py", "tests/test_oracle_l2.py"]

if __name__ == "__main__":
    with open(os.path.join(HERE, "reference_digests.json"), "w") as f:
        f.write("{}\n")
    env = dict(os.environ, NRSC5_WRITE_REF_DIGESTS="1")
    sys.exit(subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *TESTS], cwd=ROOT, env=env).returncode)
