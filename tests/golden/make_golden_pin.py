"""Generates tests/golden/golden_pin_v1.npz: the reference's side of every comparison in tests/test_reference_pin.py and
tests/test_host_pin.py, recorded from oracle/_ref/libteb_ref.so (the reference's own code, see tests/ref_binding.py) by
running those tests against the library. Run where the library can be built (next to the reference's sources):

    python -m tests.golden.make_golden_pin

Per test (key `<module>::<test name>`): `digests`, 16 bytes of SHA-256 per bit-equality check (ref_binding.digest), and
`layout` / `values` for the results compared with a tolerance. The inputs are the tests' seeded ones (not stored)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import pytest  # noqa: E402

from tests import ref_binding as rb  # noqa: E402

if __name__ == "__main__":
    rb.lib()
    rb.RECORD = {}
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_reference_pin.py"),
                      os.path.join(ROOT, "tests", "test_host_pin.py")])
    if rc != 0:
        sys.exit(f"the tests failed against the library (pytest exit code {rc}); {rb.GOLDEN_PIN} left as it was")
    data = {k: v for pins in rb.RECORD.values() for k, v in pins.arrays().items()}
    np.savez_compressed(rb.GOLDEN_PIN, **data)
    print(rb.GOLDEN_PIN, os.path.getsize(rb.GOLDEN_PIN), "bytes,", len(rb.RECORD), "tests")
