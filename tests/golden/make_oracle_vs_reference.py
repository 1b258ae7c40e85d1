"""Writes tests/golden/oracle_vs_reference.npz from the COMPILED REFERENCE (oracle/_ref, built by oracle/build_ref.sh):
the answers tests/test_oracle_vs_reference.py checks the oracle (and, where it is built, the reference) against.

    python tests/golden/make_oracle_vs_reference.py

Exact answers are stored field by field as truncated SHA-256 digests (test_oracle_vs_reference.digest), the two DCT modes
compared with a tolerance as values.  Refuses to run where the reference is not built: an answer file written from the
oracle would only pin the oracle to itself."""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import test_oracle_vs_reference as t  # noqa: E402
from oracle.pyoracle import Reference, build  # noqa: E402


def main():
    build()
    if not Reference.available():
        sys.exit("make_oracle_vs_reference.py: oracle/_ref is not built (oracle/build_ref.sh needs the reference's source tree)")
    impl = t.ReferenceAsOracle(Reference(), tempfile.mkdtemp())
    got = {}
    for fn, params in t.CASES:
        for p in params:
            got.update(fn(impl, *p))
    leaves = sorted(leaf for k, v in got.items() if k not in t.APPROX for leaf in t.leaves(k, v))
    out = {"keys": np.array([k for k, _ in leaves]),
           "digests": np.array([np.frombuffer(t.digest(a), np.uint8) for _, a in leaves])}
    out.update({f"approx/{k}": np.asarray(got[k], np.float64) for k in t.APPROX})
    path = os.path.join(HERE, "oracle_vs_reference.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(leaves)} digests + {len(t.APPROX)} value arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
