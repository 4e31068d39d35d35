#!/usr/bin/env python
"""Random-shape check of the fused bf16 path (forward, inference, backward) against the fp64 oracle.
`python tools/fuzz_fused.py [count] [seed]`; prints one line per shape, exits non-zero on a mismatch."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from tests.helpers import rel_l2  # noqa: E402
from tests.test_gpu_fused import TOL, _oracle, _params, _run  # noqa: E402
from oracle import siren_oracle as so  # noqa: E402


def main():
    count = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    bad = 0
    for it in range(count):
        d = int(rng.choice([1, 2, 3, 4, 5, 8, 11, 16]))
        nh = int(rng.integers(1, 5))
        o = int(rng.integers(1, 4))
        tasks = int(rng.choice([1, 1, 2, 3, 5]))
        per_task = bool(rng.integers(0, 2)) and tasks > 1
        n = int(rng.choice([1, 100, 128, 129, 255, 257, 384, 500, 640, 1000, 1500, 2049, 5000]))
        Ws, bs = _params(d, nh, o, tasks, per_task, seed=100 + it)
        x = so.make_coords(tasks, n, d, seed=200 + it)
        gy = (rng.standard_normal((tasks, n, o)) / n).astype(np.float32)
        yo, oW, ob = _oracle(x, Ws, bs, gy, per_task)
        y_i, _, _ = _run(x, Ws, bs, train=False)
        y_f, dW_f, db_f = _run(x, Ws, bs, train=True, gy=gy)
        errs = [rel_l2(y_i, yo), rel_l2(y_f, yo)] + [rel_l2(a, b) for a, b in zip(dW_f, oW)] + \
               [rel_l2(a, b) for a, b in zip(db_f, ob)]
        ok = max(errs) < TOL and np.isfinite(max(errs))
        bad += 0 if ok else 1
        print("%s d=%d nh=%d o=%d tasks=%d per_task=%d n=%d  vs oracle %.2e" %
              ("ok  " if ok else "FAIL", d, nh, o, tasks, per_task, n, max(errs)), flush=True)
    print("%d shapes, %d failures" % (count, bad))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
