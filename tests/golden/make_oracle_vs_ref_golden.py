"""Generates tests/golden/oracle_vs_ref_golden.json: the reference's side of every comparison in tests/test_oracle_vs_ref.py, keyed by
the pnol_ref_cli call (shape and SHA-256 of each array, values of the small ones), so that the module runs where the reference's
sources are not at hand.

    python tests/golden/make_oracle_vs_ref_golden.py

The module requires the reference to return the oracle's outputs bit for bit, so those are what is recorded here: the module is run
once with the recording switched on and the oracle's side of each check is stored. The three calls the oracle does not reproduce
bit for bit (PowerObject's run-time pow, the expcurve and cubic known answers) are taken from the reference's own outputs in
tests/golden/ref_golden.npz. Where oracle/_ref is built, the module also runs every call fresh and compares it with this recording."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main():
    out = os.path.join(HERE, "oracle_vs_ref_golden.json")
    env = dict(os.environ, PNOL_RECORD_ORACLE_VS_REF=out)
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_vs_ref.py")],
                          cwd=ROOT, env=env)
    print("wrote %s: %.1f KB" % (out, os.path.getsize(out) / 1024))


if __name__ == "__main__":
    main()
