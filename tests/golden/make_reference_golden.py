"""Writes tests/golden/reference_v1.npz from the REAL reference (d3p + jax + numpyro + jax-chacha-prng):

    python tests/golden/make_reference_golden.py            # needs the packages pinned by the reference's setup.py:46-49

The vectors (baseline/run_reference.py:dump) pin what the reference's own tests leave open (SURVEY.md section 8c):
the key-derivation rule of jax-chacha-prng, keystream word order, uniform / normal / randint transforms, Feistel and
Poisson indices, jax.random's Threefry layouts and gamma sampler, numpyro's seed plumbing (through 3-step
``DPSVI.update`` trajectories of the four example model families).  tests/test_reference_golden.py consumes the file.

``--from-oracle PATH`` writes the same file layout from the repo's own oracle instead: a format / consumer check
(tests/test_reference_golden.py::test_writer_and_consumer_roundtrip), NOT a reference — the file says so in ``impl``.
None of jax / numpyro / chacha exists in this image, so the committed tree has no reference_v1.npz: parity of those
third-party rules stays "unpinned" until this script has run somewhere they are installed.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from baseline import run_reference as rr  # noqa: E402


def main(argv):
    if len(argv) >= 2 and argv[0] == "--from-oracle":
        keys = rr.dump(rr.OracleImpl(), argv[1])
        print(f"wrote {len(keys)} arrays from the ORACLE to {argv[1]} (format check only)")
        return 0
    ok, why = rr.available()
    if not ok:
        print("reference unavailable:", why)
        return 2
    path = os.path.join(ROOT, "tests", "golden", "reference_v1.npz")
    keys = rr.dump_golden(path)
    print(f"wrote {len(keys)} arrays to {path}")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
