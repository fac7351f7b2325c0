"""Fixture arrays that a test compares bit for bit: small ones are stored as they
are, larger ones as the SHA-256 of their dtype, shape and bytes, so that
tests/golden/ stays small while the comparison stays exact."""
import hashlib

import numpy as np

LIMIT = 256  # elements; larger exact arrays are stored by digest


def array_digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def store_exact(g, key, a):
    """Put `a` into the fixture dict `g` under `key`, or its digest under `key + "_sha256"`."""
    a = np.asarray(a)
    if a.size > LIMIT:
        g[key + "_sha256"] = np.str_(array_digest(a))
    else:
        g[key] = a


def assert_exact(g, key, a, msg=""):
    """`a` equals, dtype and shape included, what store_exact recorded under `key` in `g`."""
    a = np.asarray(a)
    if key in g:
        want = g[key]
        assert a.dtype == want.dtype and np.array_equal(a, want), (key, msg)
    else:
        assert array_digest(a) == str(g[key + "_sha256"]), (key, msg)
