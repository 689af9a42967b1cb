"""Generates tests/golden/nms_lists.npz with the reference's own soft-NMS (src/lib/external/nms.pyx, compiled
by oracle/build_ref.build_nms into oracle/_ref/).  Needs the reference sources, the `cython` command on PATH,
gcc and the Python and NumPy headers; no GPU:
    python tests/golden/make_golden_nms.py

Three random box lists (70 boxes, seeded) through soft_nms with the gaussian, linear and hard methods; the
inputs, the arrays as the reference left them and the number of boxes it kept are stored.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import build_ref  # noqa: E402

CASES = ((2, 0.5), (1, 0.3), (0, 0.4))      # (method, Nt)


def main():
    ref = build_ref.load_nms()
    assert ref is not None, "the reference nms module could not be built"
    rng = np.random.default_rng(5)
    out = {}
    for i, (method, Nt) in enumerate(CASES):
        x = rng.uniform(0, 200, 70); y = rng.uniform(0, 200, 70)
        b = np.stack([x, y, x + rng.uniform(10, 90, 70), y + rng.uniform(10, 90, 70), rng.uniform(0, 1, 70)],
                     1).astype(np.float32)
        a = b.copy()
        keep = ref.soft_nms(a, Nt=Nt, method=method)
        out["in%d" % i], out["out%d" % i], out["n%d" % i] = b, a, np.int64(len(keep))
        out["cfg%d" % i] = np.array([method, Nt], np.float64)
    np.savez_compressed(os.path.join(HERE, "nms_lists.npz"), **out)
    print("wrote nms_lists", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
