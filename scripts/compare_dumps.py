"""Compare two `bench.py --dump-outputs` directories bit for bit.

    python scripts/compare_dumps.py A B

Every .npy array of A must exist in B with the same dtype, shape and raw bits (NaNs compare by their bit pattern, and
-0.0 differs from +0.0).  Prints one line per array and, for the first array that differs, the first differing env
(row) and field (column).  Exit status 0 when everything matches, 1 otherwise.  Use it to check that a change which
should not alter results (a faster kernel, a different launch shape) really computes the same outputs.
"""
import os
import sys

import numpy as np


def compare(a_dir, b_dir):
    names = sorted(f for f in os.listdir(a_dir) if f.endswith(".npy"))
    if not names:
        print("no .npy files in %s" % a_dir)
        return 1
    extra = sorted(set(f for f in os.listdir(b_dir) if f.endswith(".npy")) - set(names))
    bad = 0
    for f in names:
        pb = os.path.join(b_dir, f)
        if not os.path.exists(pb):
            print("%-20s missing in %s" % (f, b_dir))
            bad += 1
            continue
        a, b = np.load(os.path.join(a_dir, f)), np.load(pb)
        if a.dtype != b.dtype or a.shape != b.shape:
            print("%-20s dtype / shape differ: %s %s vs %s %s" % (f, a.dtype, a.shape, b.dtype, b.shape))
            bad += 1
            continue
        ua = np.ascontiguousarray(a).view(np.uint8).reshape(a.shape[0] if a.ndim else 1, -1)
        ub = np.ascontiguousarray(b).view(np.uint8).reshape(ua.shape)
        rows = np.flatnonzero((ua != ub).any(axis=1))
        if rows.size == 0:
            print("%-20s identical (%s %s)" % (f, a.dtype, a.shape))
            continue
        bad += 1
        ra, rb = a.reshape(a.shape[0], -1)[rows[0]], b.reshape(b.shape[0], -1)[rows[0]]
        col = int(np.flatnonzero(ra.view(np.uint8).reshape(ra.size, -1) != rb.view(np.uint8).reshape(rb.size, -1))[0]
                  // ra.itemsize) if ra.size > 1 else 0
        print("%-20s %d of %d envs differ; first: env row %d, field %d: %r vs %r"
              % (f, rows.size, a.shape[0], rows[0], col, ra[col], rb[col]))
    for f in extra:
        print("%-20s only in %s" % (f, b_dir))
        bad += 1
    print("identical" if bad == 0 else "%d array(s) differ" % bad)
    return 0 if bad == 0 else 1


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(compare(sys.argv[1], sys.argv[2]))
