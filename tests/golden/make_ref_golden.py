"""Records tests/golden/ref/*.npz: what the reference's compiled code (oracle/_ref/liblimap_ref.so, oracle/Makefile target
`ref`) and its own Python files return on the seeded inputs of tests/test_ref_pinning.py and tests/test_runner_dropin.py.
Those tests regenerate the same inputs and compare the oracle / the mirror with the stored outputs.

    LIMAP_REFERENCE=<LIMAP source tree> python tests/golden/make_ref_golden.py

Run from the repository root after build(), where oracle/_ref has been compiled."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

if __name__ == "__main__":
    if not os.path.isdir(os.environ.get("LIMAP_REFERENCE", "")):
        sys.exit("set LIMAP_REFERENCE to a LIMAP source tree")
    env = dict(os.environ, LIMAP_REF_RECORD="1")
    sys.exit(subprocess.call([sys.executable, "-m", "pytest", "-q", "-m", "not gpu", "tests/test_ref_pinning.py",
                              "tests/test_runner_dropin.py"], cwd=ROOT, env=env))
