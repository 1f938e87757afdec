"""Records tests/golden/ref_calls.npz: the results of every reference call the tests make through the `ref` fixture, taken from the
UNMODIFIED reference (oracle/_ref/libwelle_ref.so, built by oracle/Makefile from the reference's sources).  Run after build(), where
the reference build exists, on a machine with a B200 (test_gpu_glue.py's TII test is one of them):
    python tests/golden/make_ref_calls.py [OUT]
Elsewhere the `ref` fixture (tests/conftest.py) answers from the file (tests/refcalls.py)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.bind import Ref  # noqa: E402

TESTS = ["tests/test_oracle_vs_ref.py", "tests/test_figdb.py", "tests/test_gpu_glue.py::test_tii_spectra_tap_and_glue_measurements"]


def main():
    if not Ref.available():
        sys.exit("oracle/_ref/libwelle_ref.so is not built: nothing to record")
    out = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_calls.npz"))
    env = dict(os.environ, DABB_RECORD_REF=out)
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"] + TESTS, env=env, cwd=ROOT)
    print(f"{out}: {os.path.getsize(out)} bytes")


if __name__ == "__main__":
    main()
