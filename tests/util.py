"""Shared helpers of the parity tests."""
import hashlib
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
LIBREF = os.path.join(ROOT, "oracle", "_ref", "libsphref.so")

# north_star tolerance: <= 1e-5 relative on positions / densities after one step
TOL = 1e-5


def relerr(a, b) -> float:
    """max |a - b| relative to the scale of the reference field b (max |b|): the measure used for the
    `<= 1e-5 rel` bar.  Scale-relative (not element-wise) because force-like sums cancel in the bulk."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    scale = max(float(np.max(np.abs(b))), 1e-30)
    return float(np.max(np.abs(a - b))) / scale


def assert_close(a, b, tol=TOL, what=""):
    e = relerr(a, b)
    assert e <= tol, f"{what}: scale-relative error {e:.3e} > {tol:.1e}"


def assert_close_sample(a, gold, key, tol=TOL, what=""):
    """assert_close against a stored sample of a reference field: rows gold[<case>.idx] of `a` against gold[key],
    relative to max |b| over the WHOLE reference field (gold[key + '.scale']) -- relerr's measure on the sampled rows."""
    idx = gold[key.split(".")[0] + ".idx"]
    d = np.abs(np.asarray(a, np.float64)[idx] - np.asarray(gold[key], np.float64))
    e = float(np.max(d)) / max(float(gold[key + ".scale"]), 1e-30)
    assert e <= tol, f"{what}: scale-relative error {e:.3e} > {tol:.1e} (on {idx.size} stored rows)"


def digest(a) -> str:
    """sha256 of an array's bytes: a bit-exact comparison with a stored reference output without storing the output."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def cell_start_from_p2c(p2c, ncells):
    """fill + countingInCell_CUDA + exclusive_scan (SPHSystem.cu:123-125) on the host."""
    counts = np.bincount(p2c, minlength=ncells + 1).astype(np.int64)
    cs = np.zeros(ncells + 1, np.int64)
    cs[1:] = np.cumsum(counts)[:-1]
    return cs.astype(np.int32)
