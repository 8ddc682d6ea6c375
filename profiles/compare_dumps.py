"""Largest differences between two `bench.py --dump-outputs` directories: python profiles/compare_dumps.py A B prints
the loss difference (absolute and relative) and the three weight tensors that differ most, as a share of B's max |w|.
Used to compare a change with its parent commit next to the spread of two runs of one build."""
import sys, os, glob
import numpy as np
a, b = sys.argv[1], sys.argv[2]
worst = {}
for f in sorted(glob.glob(os.path.join(a, "*.npy"))):
    x = np.load(f).astype(np.float64); y = np.load(os.path.join(b, os.path.basename(f))).astype(np.float64)
    d = np.abs(x - y).max(); s = np.abs(y).max()
    worst[os.path.basename(f)] = (d, d / s if s else d)
l = worst.pop("loss.npy")
top = sorted(worst.items(), key=lambda kv: -kv[1][1])[:3]
print(f"{os.path.basename(a)} vs {os.path.basename(b)}: loss maxabs {l[0]:.3e} rel {l[1]:.3e}; worst weights " +
      ", ".join(f"{k} {v[0]:.2e} ({v[1]:.2e} of max)" for k, v in top))
