"""Compare the outputs two runs of `bench.py --dump-outputs DIR` wrote (same seed, same arm): for each .npy file, the largest
absolute difference and that difference over the larger of the two runs' abs-max.

    python scripts/compare_dumps.py DIR_A DIR_B [DIR_C ...]

Every further directory is compared with DIR_A.  Run the parent twice to see how far two runs of the same build differ (the
LayerNorm and BatchNorm weight gradients are column sums by float atomics, so they vary from run to run)."""
import os
import sys

import numpy as np


def compare(a, b):
    out = {}
    for name in sorted(f for f in os.listdir(a) if f.endswith(".npy")):
        x, y = np.load(os.path.join(a, name)).astype(np.float64), np.load(os.path.join(b, name)).astype(np.float64)
        d = float(np.abs(x - y).max()) if x.size else 0.0
        scale = max(float(np.abs(x).max()), float(np.abs(y).max()), 1e-30)
        out[name[:-4]] = (d, d / scale)
    return out


if __name__ == "__main__":
    if len(sys.argv) < 3:
        sys.exit(__doc__)
    base = sys.argv[1]
    for other in sys.argv[2:]:
        print(f"{base} vs {other}")
        for name, (d, r) in compare(base, other).items():
            print(f"  {name:12s} max abs diff {d:.3e}  rel to abs-max {r:.3e}")
