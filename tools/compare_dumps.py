"""Compare two `bench.py --dump-outputs` directories: decoded records and per-image counts must be identical, and the sampled
logits equal (bit for bit by default, or within --atol).

    python tools/compare_dumps.py DIR_A DIR_B [--atol 0]

Prints one JSON line with the result and exits non-zero on a difference."""
import argparse
import glob
import json
import os
import sys

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--atol", type=float, default=0.0)
    args = ap.parse_args()
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(args.a, "*.npy")))
    if sorted(os.path.basename(p) for p in glob.glob(os.path.join(args.b, "*.npy"))) != names or not names:
        print(json.dumps({"equal": False, "error": "the two directories hold different files"}))
        return 1
    report, ok = {}, True
    for name in names:
        x, y = np.load(os.path.join(args.a, name)), np.load(os.path.join(args.b, name))
        if x.shape != y.shape:
            report[name] = {"shape_a": list(x.shape), "shape_b": list(y.shape)}
            ok = False
            continue
        diff = float(np.max(np.abs(x.astype(np.float64) - y.astype(np.float64)))) if x.size else 0.0
        tolerant = name.startswith("logits_") and args.atol > 0
        same = diff <= args.atol if tolerant else bool(np.array_equal(x, y))
        report[name] = {"rows": int(x.shape[0]), "max_abs_diff": diff, "equal": same}
        ok &= same
    print(json.dumps({"equal": ok, "files": report}))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
