"""Bit-exact fingerprint of an array for the goldens: [shape, dtype, SHA-256 of the C-contiguous bytes].  Two arrays have the same digest
exactly when they have the same shape, dtype and bits, so a stored digest stands in for a stored array in a bit-identity check."""
import hashlib

import numpy as np


def digest(a):
    """a: numpy array or torch tensor"""
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a)
    return [list(a.shape), str(a.dtype), hashlib.sha256(a.tobytes()).hexdigest()]
