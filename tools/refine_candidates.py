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


F32, F64 = np.float32, np.float64


def _fma(a, b, c):
    """float32 fma: the product is exact in float64, the sum is rounded twice (close enough for a model)"""
    return (np.asarray(a, F64) * np.asarray(b, F64) + np.asarray(c, F64)).astype(F32)


def _approx(v, sign):
    """rsqrt.approx / sqrt.approx, pushed by 2^-22 in the direction that hurts the bound (sign -1: smaller)"""
    return (np.asarray(v, F64) * (1.0 + sign * 2.0 ** -22)).astype(F32)


def kernel_bound(li, y0, y1, y2, xs):
    """refine.cu's bound (the note above refine_kernel), in its float32 arithmetic, for left stacks li and right stacks
    y0, y1, y2 (integer arrays [n, pixels]) at the steps xs: (wraps [pixels], ub [steps, pixels], rho [steps, pixels]).
    ub is 2 where the kernel has no bound."""
    n = li.shape[0]
    y0, y1, y2, li = (np.asarray(v, np.int64) for v in (y0, y1, y2, li))
    a = (F32(0.5) * (y0 - 2 * y1 + y2).astype(F32)).astype(F64)
    b = (F32(0.5) * (y2 - y0).astype(F32)).astype(F64)
    t2 = 4 * a * a - b * b  # exact: quarters below 2^24
    t1 = b * b - 510 * np.abs(a) - 4 * a * (y1 - 127.5)
    wraps = np.minimum(t1, t2).max(0) > 0

    def N(u, v):
        return n * (u * v).sum(0) - u.sum(0) * v.sum(0)

    A, B, C = y0 - 2 * y1 + y2, y2 - y0, y1
    nBB, nAC = N(B, B).astype(F32), N(A, C).astype(F32)
    e = [N(C, C).astype(F32), N(B, C).astype(F32), _fma(nBB, 0.25, nAC),
         F32(0.5) * N(A, B).astype(F32), F32(0.25) * N(A, A).astype(F32)]
    m = [N(li, C).astype(F32), F32(0.5) * N(li, B).astype(F32), F32(0.5) * N(li, A).astype(F32)]
    ev = F32(2.0 ** -20) * (np.abs(e[0]) + np.abs(e[1]) + F32(0.25) * np.abs(nBB) + np.abs(nAC) + np.abs(e[3])
                            + np.abs(e[4]))
    ec = F32(2.0 ** -21) * (np.abs(m[0]) + np.abs(m[1]) + np.abs(m[2]))
    var0 = N(li, li).astype(F32)
    with np.errstate(divide="ignore", invalid="ignore"):
        r0 = _approx(1.0 / np.sqrt(var0.astype(F64)), -1) * F32(1.0 + 2.0 ** -18)
        hn = F32(n) * F32(0.5 + 2.0 ** -9)
        ubs, rhos = [], []
        for x in np.asarray(xs, F32):
            v = _fma(_fma(_fma(_fma(e[4], x, e[3]), x, e[2]), x, e[1]), x, e[0]) - ev
            c = _fma(_fma(m[2], x, m[1]), x, m[0]) + ec
            y = _approx(1.0 / np.sqrt(np.where(v > 0, v, np.nan).astype(F64)), -1)
            s = hn * y
            rho = np.minimum(F32(1), np.maximum(F32(0), (c * r0) * y))
            cu = _fma(F32(-0.5) * s, s, F32(1))
            r = _approx(np.sqrt(_fma(-rho, rho, F32(1)).astype(F64)), -1)
            ub = np.where(rho >= cu, F32(2), _fma(rho, cu, _fma(r, s, F32(2.0 ** -19))))
            ub = np.where((v > 0) & (s < 1), ub, F32(2))
            ubs.append(ub)
            rhos.append(np.nan_to_num(rho, nan=0.0))
    return wraps, np.stack(ubs).astype(F64), np.stack(rhos)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frame", type=int, default=0)
    ap.add_argument("--row0", type=int, default=760)
    ap.add_argument("--rows", type=int, default=16)
    ap.add_argument("--margin", type=float, default=(4 * N + 40) * 2.0 ** -24)
    ap.add_argument("--bound", action="store_true")
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
    out = {
        "frame": args.frame, "rows": [args.row0, args.row0 + args.rows - 1], "pixels": int(count.size),
        "margin": args.margin, "candidates": hist,
        "share": {k: v / max(count.size, 1) for k, v in hist.items()},
        "gap_best_second_p01": float(np.quantile(gap, 0.01)) if gap.size else None,
    }
    if args.bound:
        out.update(bound_stats(li, *(v.astype(np.int64) for v in (y0, y1, y2)), s, r, c, cols, args.margin))
    print(json.dumps(out))


def survivors(ub, rho, wraps, s, margin):
    """A pruned screen's rounds: the two steps of largest rho first, then, in step order, the steps whose bound reaches
    the floor. The floor here is the one after the first round; the kernel's rises with every round, so these
    counts are an upper bound. The exact scores s stand in for the screened ones. Returns (survivors, rounds)."""
    nsteps, npx = ub.shape
    order = np.argsort(-rho, axis=0, kind="stable")
    first = order[:2]
    s_first = np.take_along_axis(s, first, 0).max(0)
    floor = np.maximum(s_first, -1.0) - margin
    keep = (ub >= floor) | wraps[None, :]
    keep[first, np.arange(npx)] = False
    rest = keep.sum(0)
    return rest + min(2, nsteps), 1 + (rest + 1) // 2


def bound_stats(li, y0, y1, y2, s, r, c, cols, margin):
    xs = steps(CFG["subpixel_step"])
    wraps, ub, rho = kernel_bound(li, y0, y1, y2, xs)
    ok = wraps | ((ub >= s - 1e-12) | ~np.isfinite(s)).all(0)  # the bound holds wherever it applies
    assert ok.all(), f"{(~ok).sum()} pixels with a score above its bound"
    surv, rounds = survivors(ub, rho, wraps, s, margin)
    warp = r.astype(np.int64) * ((cols + 31) // 32) + c // 32  # lanes of a warp: 32 consecutive columns
    _, inv = np.unique(warp, return_inverse=True)
    per_warp = np.zeros(inv.max() + 1, np.int64)
    np.maximum.at(per_warp, inv, rounds)
    return {
        "steps": len(xs), "wrap_share": float(wraps.mean()),
        "survivors_per_pixel": {"mean": float(surv.mean()), "median": float(np.median(surv)),
                                "p90": float(np.quantile(surv, 0.9)), "max": int(surv.max())},
        "rounds_per_warp": {"mean": float(per_warp.mean()), "unpruned": (len(xs) + 1) // 2},
    }


if __name__ == "__main__":
    main()
