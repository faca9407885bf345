"""Golden arrays of tests/golden/independent.npz that are stored pinned rather than in full (the kNN and
cv2.flann radius lists): the SHA-256 of the whole array, which pins it bit for bit, and its rows at a
seeded sample (tests/golden/make_golden.py)."""
import hashlib

import numpy as np


def assert_pinned(golden, key, got):
    """got equals the pinned golden `key` bit for bit.  The sampled rows are compared first so that a
    mismatch shows where; the digest then covers every row."""
    rows = golden[key + "_rows"]
    assert np.array_equal(got[rows].view(np.uint32), golden[key + "_sample"].view(np.uint32)), key
    assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == str(golden[key + "_sha256"]), key
