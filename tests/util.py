import hashlib

import numpy as np

# arrays up to this size are stored whole in the golden files; larger ones as a digest
GOLDEN_INLINE_BYTES = 16 << 10


def digest(a):
    """SHA-256 of an array's shape and values.  Integers hash as int64 and floats as float64 with every NaN made one NaN
    and -0.0 made 0.0, so two arrays have the same digest exactly when np.array_equal(a, b, equal_nan=True) holds."""
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = a.astype(np.float64)
        a = np.where(np.isnan(a), np.nan, a + 0.0)
    else:
        a = a.astype(np.int64)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def fingerprint(a):
    """What a golden file keeps of an array: the array itself when it is small, its digest() otherwise."""
    a = np.asarray(a)
    return a.copy() if a.nbytes <= GOLDEN_INLINE_BYTES else np.str_(digest(a))


def same(a, stored):
    """Whether `a` is the array a golden file kept as `stored` (see fingerprint): np.array_equal, NaN equal to NaN."""
    stored = np.asarray(stored)
    if stored.dtype.kind == "U":
        return digest(a) == str(stored)
    a = np.asarray(a)
    return a.shape == stored.shape and bool(np.array_equal(a, stored, equal_nan=a.dtype.kind == "f"))


def bits_equal(a, b):
    """Bit-for-bit equality of float64 arrays (NaN == NaN when the payload matches or both NaN)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return bool(((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))).all())


def pose_error(Xa, Xb):
    """(rotation angle [rad], translation distance [m]) between two 3x4 / 4x4 poses."""
    Xa, Xb = np.asarray(Xa)[:3], np.asarray(Xb)[:3]
    dR = Xa[:, :3] @ Xb[:, :3].T
    # atan2 form: arccos((tr-1)/2) has a ~2e-8 rad noise floor near the identity
    s = 0.5 * np.linalg.norm([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    ang = float(np.arctan2(s, (np.trace(dR) - 1.0) / 2.0))
    return ang, float(np.linalg.norm(Xa[:, 3] - Xb[:, 3]))


# north_star tolerances
POSE_RAD, POSE_M = 1e-5, 1e-4
# H/b: relative to the largest |entry| (the CPU sums ~1e5 terms sequentially; SURVEY 8d asks 1e-12)
HB_REL = 1e-12
