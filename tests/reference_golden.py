"""What the UNMODIFIED reference computed for the suite's comparisons with it, stored in tests/golden/reference_golden.json
so that those comparisons run on any checkout, without the reference sources or oracle/_ref.

Each entry is either the reference's result itself (when it is small) or the SHA-256 of a canonical encoding of everything
the comparison looked at (Digest below).  A test feeds its own side through the same encoding and compares.  The file is
written by tests/golden/make_reference_golden.py where oracle/_ref is built; it calls each test module's
reference_golden(), which computes the reference's side of that module's comparisons."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.json")
_GOLD = None


def expected(key):
    global _GOLD
    if _GOLD is None:
        with open(PATH) as f:
            _GOLD = json.load(f)
    return _GOLD[key]


class Digest:
    """SHA-256 over a canonical encoding.  Numbers compare by value, as == does: ints and floats of any width encode the
    same, and a zero encodes without its sign (encode float(x).hex() strings where the sign of zero matters).  Arrays
    encode their shape and their values as float64."""

    def __init__(self, *xs):
        self.h = hashlib.sha256()
        self.add(*xs)

    def add(self, *xs):
        for x in xs:
            self._add(x)
        return self

    def _add(self, x):
        u = self.h.update
        if isinstance(x, np.ndarray):
            a = np.ascontiguousarray(x, dtype=np.float64) + 0.0
            u(b"A%r:" % (a.shape,))
            u(a.tobytes())
        elif isinstance(x, (list, tuple)):
            u(b"[%d:" % len(x))
            for y in x:
                self._add(y)
        elif isinstance(x, dict):
            u(b"{%d:" % len(x))
            for k in sorted(x):
                self._add(k)
                self._add(x[k])
        elif isinstance(x, (bool, np.bool_, int, np.integer, float, np.floating)):
            u(b"n" + (float(x) + 0.0).hex().encode() + b";")
        elif isinstance(x, str):
            b = x.encode()
            u(b"s%d:" % len(b) + b)
        elif x is None:
            u(b"N")
        else:
            raise TypeError(type(x))

    def hexdigest(self):
        return self.h.hexdigest()


def digest(*xs):
    return Digest(*xs).hexdigest()
