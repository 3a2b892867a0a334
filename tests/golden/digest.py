"""Content digests of arrays too large to store: the golden files keep the SHA-256 of what the original project computed,
and a test recomputes it over its own result (an exact comparison)."""
import hashlib

import numpy as np


def digest(a):
    """SHA-256 over dtype, shape and the C-order bytes of `a`."""
    a = np.ascontiguousarray(np.asarray(a))
    h = hashlib.sha256(('%s %s|' % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def lists_digest(lists):
    """(lengths int32 [n], digest of the concatenation) of a list of int32 index lists, e.g. one neighbour list per point."""
    lens = np.array([len(x) for x in lists], np.int32)
    cat = np.concatenate([np.asarray(x, np.int32) for x in lists]) if len(lists) else np.zeros(0, np.int32)
    return lens, digest(cat)
