"""Writes tests/golden/reference_cases.npz, the stored record of the reference-side results of every case of
tests/test_oracle_vs_reference.py (see that module).  In a checkout without oracle/_ref/libmlpp_ref.so the tests compare
the oracle port against this record.

    python tests/golden/make_reference_cases.py            # the reference's own code: needs oracle/_ref (make -C oracle ref)
    python tests/golden/make_reference_cases.py --oracle   # the oracle port, where the reference is not available

The `source` entry of the file names what wrote it.  A record written by the oracle pins the port against later changes;
wherever oracle/_ref is built, the tests also check the record against the reference's own results."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from tests import test_oracle_vs_reference as cases  # noqa: E402


def main():
    impl = "oracle" if "--oracle" in sys.argv[1:] else "reference"
    assert impl == "oracle" or oracle.ref_available(), "build oracle/_ref first (make -C oracle ref), or pass --oracle"
    record = {"source": np.array(impl)}
    for name, run in cases.CASES.items():
        record.update(cases.record_entries(name, run(impl)))
    np.savez_compressed(cases.RECORD_PATH, **record)
    print(f"{len(cases.CASES)} cases from the {impl} into {cases.RECORD_PATH} ({os.path.getsize(cases.RECORD_PATH)} bytes)")


if __name__ == "__main__":
    main()
