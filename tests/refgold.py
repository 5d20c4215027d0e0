"""Stored outputs of the reference's own CUDA kernels, for the GPU parity tests.

The reference extensions (its bev_pool, voxel_layer and sparse_conv_ext modules compiled unmodified for
sm_100 by oracle/build_ref.py) exist only where the reference sources are, so what they returned on the
tests' seeded inputs is recorded once on a B200 by tests/golden/make_golden_gpu.py into
tests/golden/refgpu_<case>.npz, and the tests compare against that record:

  * an output the tests require to be bit-identical is stored as the SHA-256 of its dtype, shape and bytes
    (integers widened to int64);
  * an output compared within a tolerance is stored as a fixed, seeded sample of its elements plus the
    largest magnitude of the whole output (the scale of the relative bound), its shape and its NaN count.
"""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE = 2048


def _np(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a)


def digest(a):
    a = _np(a)
    if a.dtype.kind in "iu":                 # an index is the same index in int32 or int64
        a = a.astype(np.int64)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_index(n, k=SAMPLE):
    """k flat positions out of n, the same for every array of n elements."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(n).choice(n, k, replace=False))


def sample(a):
    flat = _np(a).reshape(-1)
    return flat[sample_index(flat.size)]


def path(case):
    return os.path.join(GOLDEN, "refgpu_%s.npz" % case)


class Record:
    """What one test case's reference calls returned; written by make_golden_gpu.py."""

    def __init__(self):
        self.arrays = {}

    def exact(self, key, a):
        self.arrays[key + ".sha256"] = np.array(digest(a))

    def close(self, key, a):
        a = _np(a)
        self.arrays[key + ".shape"] = np.array(a.shape, np.int64)
        self.arrays[key + ".scale"] = np.array(float(np.nanmax(np.abs(a))) if a.size else 0.0)
        self.arrays[key + ".nans"] = np.array(int(np.isnan(a).sum()))
        self.arrays[key + ".sample"] = sample(a)

    def value(self, key, v):
        self.arrays[key] = np.asarray(v)

    def save(self, case):
        np.savez_compressed(path(case), **self.arrays)


class Gold:
    """The stored record of one case, with the comparisons the tests make against it."""

    def __init__(self, case):
        with np.load(path(case)) as z:
            self.arrays = {k: z[k] for k in z.files}

    def __getitem__(self, key):
        return self.arrays[key]

    def exact(self, key, got):
        assert digest(got) == str(self.arrays[key + ".sha256"]), "%s differs from the reference" % key

    def scale(self, key):
        return float(self.arrays[key + ".scale"])

    def sample(self, key):
        return self.arrays[key + ".sample"]

    def close(self, key, got, rtol):
        """max |got - reference| over the stored sample <= rtol * max |reference| over the whole output"""
        got = _np(got)
        assert tuple(got.shape) == tuple(self.arrays[key + ".shape"]), key
        assert int(np.isnan(got).sum()) == int(self.arrays[key + ".nans"]), "%s: NaN count differs" % key
        err = np.abs(sample(got).astype(np.float64) - self.sample(key).astype(np.float64)).max(initial=0.0)
        assert err <= rtol * self.scale(key), "%s: %.3g > %g * %.3g" % (key, err, rtol, self.scale(key))
