"""Compare two directories written by `bench.py --dump-outputs`, array by array: dtype, shape, whether the two are bit for
bit equal, and the largest absolute difference over the largest magnitude in B.  Exits 1 if the sets of arrays or their shapes differ.

  python tools/compare_dumps.py DIR_A DIR_B"""
import os
import sys

import numpy as np


def main(a, b):
    names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
    other = sorted(f for f in os.listdir(b) if f.endswith(".npy"))
    if names != other:
        print("different arrays: %s vs %s" % (names, other))
        return 1
    for f in names:
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        if x.shape != y.shape:
            print("%s: shape %s vs %s" % (f, x.shape, y.shape))
            return 1
        rel = float(np.abs(x - y).max() / max(float(np.abs(y).max()), 1e-300))
        print("%-26s %-8s %-14s equal=%-5s maxrel=%.3e" % (f, x.dtype, x.shape, np.array_equal(x, y), rel))
    return 0


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
