#!/usr/bin/env python
"""Records tests/golden/reference_pins.npz (see tests/golden/pins.py): runs the tests that take the `reference`
fixture with oracle/_ref built and stores the CRC-32 of every value they compare, computed by the reference.

    python tests/golden/make_pins.py [--out FILE] [pytest arguments, e.g. -m "not gpu"]

Pins of tests that are not run keep their recorded values.  The GPU tests among them record on a machine with a
GPU; --out writes the merged file elsewhere.
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.golden import pins  # noqa: E402


def main(argv):
    out = pins.PATH
    if argv[:1] == ["--out"]:
        out, argv = argv[1], argv[2:]
    merged = dict(pins.stored())
    pins.RECORDING = {}
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests")] + argv)
    if rc != 0:
        sys.exit("tests failed; nothing written")
    merged.update({k: np.array(v, np.uint32) if isinstance(v, list) else v for k, v in pins.RECORDING.items()})
    np.savez_compressed(out, **merged)
    print("wrote %s: %d tests, %d values" % (out, len(merged), sum(len(v) for v in merged.values())))


if __name__ == "__main__":
    main(sys.argv[1:])
