"""Recorded outputs of the reference build for the tests that compare with it.

A test that compares a result with the reference takes the `reference` fixture and passes every compared value
through `reference.check(got, want)`.  Where oracle/_ref is built, `want` is computed by the reference library
(`reference.lib`), must equal `got`, and its CRC-32 must equal the one recorded for that comparison.  Where it is not
(a clean checkout: the reference sources are not part of the repository), `reference.lib` is None, `want` is not
computed and `got` must hit the recorded CRC-32 instead, so the comparison with the reference still runs.

The CRC-32s live in tests/golden/reference_pins.npz, one array per test in the order the test compares, next to the
few arrays tests take from the reference as inputs (`reference.value`); tests/golden/make_pins.py records them from
the reference build.
"""
import os
import zlib

import numpy as np

from tests import oracle_lib

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_pins.npz")
OUT = object()          # placeholder for the output array in Reference.out()
RECORDING = None        # test id -> list of CRC-32 (test id::name -> array) while make_pins.py runs
_stored = None


def digest(v):
    """CRC-32 of a compared value that does not depend on integer or float widths: arrays (and scalars) by shape and
    values, tuples / lists / dicts by their parts in order (dicts by sorted key)."""
    if isinstance(v, dict):
        v = [v[k] for k in sorted(v)]
    if isinstance(v, (tuple, list)):
        c = zlib.crc32(b"seq%d" % len(v))
        for x in v:
            c = zlib.crc32(digest(x).to_bytes(4, "little"), c)
        return c
    a = np.asarray(v)
    a = np.ascontiguousarray(a.astype(np.float64 if a.dtype.kind == "f" else np.int64))
    return zlib.crc32(a.tobytes(), zlib.crc32(repr(a.shape).encode()))


def stored():
    global _stored
    if _stored is None:
        _stored = dict(np.load(PATH)) if os.path.exists(PATH) else {}
    return _stored


class Reference:
    """The reference outputs one test compares with (see the module docstring)."""

    def __init__(self, test_id):
        self.id = test_id
        self.lib = oracle_lib.load_ref()
        self.i = 0
        if RECORDING is not None:
            assert self.lib is not None, "recording needs oracle/_ref"
            self.pins = RECORDING.setdefault(test_id, [])
            del self.pins[:]
        else:
            self.pins = stored().get(test_id)
            assert self.pins is not None, ("no recorded reference outputs for %s: run tests/golden/make_pins.py where "
                                           "oracle/_ref is built" % test_id)

    def check(self, got, want=None, msg=None):
        """`got` must equal what the reference computes: `want`, or `want(lib)` when it is callable (only called
        where the reference library is present)."""
        if self.lib is not None:
            if callable(want):
                want = want(self.lib)
            assert digest(got) == digest(want), (msg, "differs from the reference")
            d = digest(want)
        else:
            d = digest(got)
        if RECORDING is not None:
            self.pins.append(d)
        else:
            assert self.i < len(self.pins), (msg, "more comparisons than were recorded for " + self.id)
            assert d == int(self.pins[self.i]), (msg, "differs from the recorded reference output #%d" % self.i)
        self.i += 1

    def value(self, name, want):
        """An array the test takes from the reference as an input: `want(lib)` where the reference library is present
        (it must equal the recorded array), else the recorded array."""
        key = self.id + "::" + name
        if self.lib is None:
            return stored()[key]
        v = np.asarray(want(self.lib))
        if RECORDING is not None:
            RECORDING[key] = v
        else:
            assert np.array_equal(v, stored()[key]), ("differs from the recorded reference value", key)
        return v

    def out(self, got, name, *args, msg=None):
        """Checks `got` against the reference function `name` called with `args`, OUT standing for an output array
        shaped like `got`."""
        def want(lib):
            w = np.zeros_like(got)
            getattr(lib, name)(*[oracle_lib.addr(w) if a is OUT else a for a in args])
            return w
        self.check(got, want, msg)

    def finish(self):
        if RECORDING is None:
            assert self.i == len(self.pins), "%s compared %d values, %d were recorded" % (self.id, self.i, len(self.pins))
