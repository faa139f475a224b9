"""Compare two `bench.py --dump-outputs` directories: max |a - b| and the number of differing elements per array.
Usage: python profiles/compare_dumps.py DIR_A DIR_B [LABEL]  (prints one JSON line)"""
import json
import os
import sys

import numpy as np

a_dir, b_dir = sys.argv[1], sys.argv[2]
rep = {"label": sys.argv[3] if len(sys.argv) > 3 else f"{a_dir} vs {b_dir}"}
for f in sorted(os.listdir(a_dir)):
    if not f.endswith(".npy"):
        continue
    a, b = np.load(os.path.join(a_dir, f)).astype(np.float64), np.load(os.path.join(b_dir, f)).astype(np.float64)
    d = np.abs(a - b)
    rep[f[:-4]] = {"max_abs_diff": float(d.max()), "n_diff": int((d > 0).sum()), "n": int(d.size),
                   "max_abs": float(np.abs(b).max())}
print(json.dumps(rep))
