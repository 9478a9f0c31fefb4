"""Writes tests/golden/blur_oracle.npz: the CPU oracle's Gaussian taps and blurred images for the
outline-blur cases of tests/test_oracle.py.

These are the ORACLE's values (tbref_gaussian_kernel, tbref_blur_argb32), not the reference's:
the reference's gstttmlblur.c is not part of this repository and was not available to run when
the file was written. The tests compare the frozen values with numpy restatements of the
Gaussian and of pixman's convolution filter; the comparison with the reference's own code is
made by the tests that need oracle/_ref. Where oracle/_ref is built, this script refuses to write
unless the reference's code gives the same values.

The file is frozen by hash (BLUR_ORACLE_SHA256 in tests/test_oracle.py). Re-run only on purpose,
then update that hash:  python tests/golden/gen_blur_oracle.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import oracle  # noqa: E402

KERNEL_CASES = [(0, 0.7), (1, 0.5), (2, 1.0), (3, 1.5), (5, 2.5), (8, 4.0), (12, 3.3), (20, 10.0), (32, 8.0)]
BLUR_CASES = [(1, 1, 0.8), (2, 2, 1.0), (3, 4, 2.0), (4, 7, 3.0)]      # (seed, radius, sigma)


def blur_input(seed):
    """A 37 x 53 premultiplied ARGB32 image (the same as the reference tests draw)."""
    r = np.random.default_rng(seed)
    a = r.integers(0, 256, (37, 53, 1), dtype=np.uint8)
    return np.concatenate([(r.integers(0, 256, (37, 53, 3)) * a // 255).astype(np.uint8), a], axis=2)


def main():
    ref = oracle.load_ref() is not None
    data = {"source": np.array("oracle/ttmlblend_ref.c (tbref_gaussian_kernel, tbref_blur_argb32)"),
            "kernel_cases": np.array(KERNEL_CASES, dtype=np.float64),
            "blur_cases": np.array(BLUR_CASES, dtype=np.float64)}
    for k, (radius, sigma) in enumerate(KERNEL_CASES):
        data[f"taps{k}"] = oracle.gaussian_kernel(radius, sigma).ravel()
        if ref:
            assert np.array_equal(oracle.ref_blur_argb32(np.zeros((3, 3, 4), np.uint8), radius, sigma)[1][2:],
                                  data[f"taps{k}"]), (radius, sigma)
    for k, (seed, radius, sigma) in enumerate(BLUR_CASES):
        img = blur_input(seed)
        data[f"blur_in{k}"] = img
        data[f"blur_taps{k}"] = oracle.gaussian_kernel(radius, sigma).ravel()
        data[f"blur_out{k}"] = oracle.blur_argb32(img, radius, sigma)
        if ref:
            assert np.array_equal(oracle.ref_blur_argb32(img, radius, sigma)[0], data[f"blur_out{k}"]), seed
    out = os.path.join(HERE, "blur_oracle.npz")
    np.savez_compressed(out, **data)
    h = hashlib.sha256()
    for key in sorted(data):
        h.update(key.encode())
        h.update(np.ascontiguousarray(data[key]).tobytes())
    print("wrote", out, "(checked against oracle/_ref)" if ref else "(oracle/_ref not built: not checked "
          "against the reference)", "sha256", h.hexdigest())


if __name__ == "__main__":
    main()
