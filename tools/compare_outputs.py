"""Compare the arrays `bench.py --dump-outputs` wrote for two builds against the spread of one build with itself.

    python tools/compare_outputs.py BASE_DIR1 BASE_DIR2 [...] -- NEW_DIR1 [...]

The dumps of the base build (at least two runs) give its run-to-run spread per array: split-K GEMMs accumulate with fp32 atomics in no
fixed order, so two runs of one build already differ a little.  Every new run must stay within `--allow` times that spread of every
base run.  Per array: the largest absolute difference and the relative L2 difference.  Exit code 1 if an array is outside."""
import argparse
import itertools
import os
import sys

import numpy as np

NAMES = ["loss", "global_grad_norm", "params", "master_params", "exp_avg", "exp_avg_sq"]


def diff(a, b):
    a = a.astype(np.float64); b = b.astype(np.float64)
    return float(np.abs(a - b).max()), float(np.linalg.norm(a - b) / max(np.linalg.norm(a), 1e-30))


def main():
    argv = sys.argv[1:]
    if "--" not in argv:
        sys.exit(__doc__)
    i = argv.index("--")
    ap = argparse.ArgumentParser()
    ap.add_argument("--allow", type=float, default=2.0)
    opts, base = ap.parse_known_args(argv[:i])
    new = argv[i + 1:]
    if len(base) < 2 or not new:
        sys.exit("need two or more base dumps and one or more new dumps")
    load = lambda d: {n: np.load(os.path.join(d, n + ".npy")) for n in NAMES}
    B, N = [load(d) for d in base], [load(d) for d in new]
    ok = True
    for n in NAMES:
        spread = [diff(x[n], y[n]) for x, y in itertools.combinations(B, 2)]
        s_abs, s_rel = max(s[0] for s in spread), max(s[1] for s in spread)
        got = [diff(x[n], b[n]) for x in N for b in B]
        g_abs, g_rel = max(g[0] for g in got), max(g[1] for g in got)
        good = g_abs <= opts.allow * s_abs and g_rel <= opts.allow * s_rel
        ok &= good
        print(f"{n:17s} base-vs-base max|d| {s_abs:.3e} rel-L2 {s_rel:.3e} | new-vs-base max|d| {g_abs:.3e} rel-L2 {g_rel:.3e} | "
              f"{'ok' if good else 'OUTSIDE'} (allow x{opts.allow:g})" + (f"  value {float(B[0][n][0]):.6f}" if B[0][n].size == 1 else ""))
    print("all arrays within the base spread" if ok else "SOME ARRAYS OUTSIDE THE BASE SPREAD")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
