#!/usr/bin/env python
"""How many subpixel steps per pixel the uint8 refine screen keeps as candidates, on the CPU.

For rows of a bench frame (libbicos_b200/synth.py, the bench workload's config) the oracle gives the raw disparities;
for every refined non-border pixel this computes, with the reference's float32 interpolation, the exact correlation
of every x step from integer moments, and counts the steps within a margin of max(-1, best): the steps the kernel
would run through the float chain (refine.cu, the note above refine_kernel). Pixels with more than two candidates
take the unscreened loop. Prints one JSON line.

    python tools/refine_candidates.py [--frame 0] [--row0 760] [--rows 16] [--margin 2e-5]

--margin defaults to the kernel's screen_margin(33) = (4 * 33 + 40) * 2^-24.
"""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from libbicos_b200 import synth  # noqa: E402

N, HEIGHT, WIDTH = 33, 1536, 2048
CFG = dict(min_variance=2.0, subpixel_step=0.1, max_lr_diff=1)  # bench.py CFG


def steps(step):
    xs, x = [], np.float32(-1.0)
    while x <= np.float32(1.0):  # the reference's float loop
        xs.append(x)
        x = np.float32(x + np.float32(step))
    return np.array(xs, dtype=np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frame", type=int, default=0)
    ap.add_argument("--row0", type=int, default=760)
    ap.add_argument("--rows", type=int, default=16)
    ap.add_argument("--margin", type=float, default=(4 * N + 40) * 2.0 ** -24)
    args = ap.parse_args()

    oracle.build(ref=False)
    left, right, _ = synth.make_stacks(N, HEIGHT, WIDTH, np.uint8, frame=args.frame, row0=args.row0, rows=args.rows)
    port = oracle.port
    d0 = port.descriptors(left, False, wide=True)
    d1 = port.descriptors(right, False, wide=True)
    raw = port.bicos(d0, d1, oracle.FLAG_CONSISTENCY, CFG["max_lr_diff"]).astype(np.int64)

    rows, cols = raw.shape
    r, c = np.nonzero(raw != -32768)
    c1 = c - raw[r, c]
    keep = (c1 > 0) & (c1 < cols - 1)  # in the image and not on its border
    r, c, c1 = r[keep], c[keep], c1[keep]
    li = left[:, r, c].astype(np.int64)  # [n, pixels]
    y0, y1, y2 = (right[:, r, c1 + k].astype(np.float32) for k in (-1, 0, 1))
    qa = np.float32(0.5) * ((y0 - np.float32(2.0) * y1) + y2)
    qb = np.float32(0.5) * (y2 - y0)

    n = N
    sl, sll = li.sum(0), (li * li).sum(0)
    var0 = n * sll - sl * sl
    minvar_n = np.float32(CFG["min_variance"]) * np.float32(n)  # float var is var_n / n; compared with min_variance * n
    scores = []
    for x in steps(CFG["subpixel_step"]):
        v = ((qa * x) * x + qb * x) + y1  # five separately rounded float32 operations
        v = (np.rint(v).astype(np.int64)) & 0xFF  # roundevenf, then the wrap to uint8
        sv, svv, slv = v.sum(0), (v * v).sum(0), (li * v).sum(0)
        var1 = n * svv - sv * sv
        cov = n * slv - sl * sv
        with np.errstate(divide="ignore", invalid="ignore"):
            rho = cov / np.sqrt(var0.astype(np.float64) * var1)
        # NaN (a zero variance) and the exact -1 of a small variance cannot win
        rho[(var1 == 0) | (var0 == 0) | (var1 < n * minvar_n) | (var0 < n * minvar_n)] = -np.inf
        scores.append(rho)
    s = np.stack(scores)  # [steps, pixels]
    floor = np.maximum(s.max(0), -1.0) - args.margin
    count = (s >= floor).sum(0)
    s_sorted = np.sort(s, axis=0)
    gap = (s_sorted[-1] - s_sorted[-2])[np.isfinite(s_sorted[-2])]
    hist = {str(k): int((count == k).sum()) for k in range(int(count.max()) + 1)}
    print(json.dumps({
        "frame": args.frame, "rows": [args.row0, args.row0 + args.rows - 1], "pixels": int(count.size),
        "margin": args.margin, "candidates": hist,
        "share": {k: v / max(count.size, 1) for k, v in hist.items()},
        "gap_best_second_p01": float(np.quantile(gap, 0.01)) if gap.size else None,
    }))


if __name__ == "__main__":
    main()
