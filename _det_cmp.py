import os, sys
import numpy as np
a, b = sys.argv[1:3]
rows, same = [], 0
for f in sorted(os.listdir(a)):
    x, y = np.load(os.path.join(a, f)).astype(np.float64), np.load(os.path.join(b, f)).astype(np.float64)
    same += np.array_equal(x, y)
    scale = max(np.abs(y).max(), 1e-30) if y.size else 1.0
    d = np.abs(x - y)
    rows.append((float(d.max() / scale) if d.size else 0.0, int((d > 1e-5 * scale).sum()), f))
rows.sort(reverse=True)
print(len(rows), "arrays,", same, "bit-identical; worst (max|diff|/max|ref|, elements beyond 1e-5 of scale, name):")
for r in rows[:8]:
    print("  ", r)
