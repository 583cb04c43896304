"""The refine stage on its own (refine.cu, `Handle.refine`), bit for bit against the oracle's agree(), on keys chosen
per pixel instead of keys found by a search.

Every pixel of a scene is a left stack refined against a right triple (columns col1 - 1, col1, col1 + 1) that the test
chose, so that the cases the subpixel screen's proof rests on (the note above refine_kernel) occur on purpose and
densely:
  * interp: the left stack is the kernel's rounded interpolation of the triple at a grid step, at the midpoint of two
    grid steps or at a random x, sometimes with +-1 noise; winners at the first and the last grid step;
  * wrap: triples whose parabola leaves the input range (the left stack is the WRAPPED interpolation at an overshooting
    step), touches its end exactly (t1 = 0), overshoots by less than 1/2, or has its vertex exactly at x = +-1 (t2 = 0);
  * mined: interp pixels whose float winner is not the exact argmax, or with two or with three or more steps within
    screen_margin(n) of the best exact score;
  * flat: nearly constant and constant triples, a constant left stack, a left stack of the smallest nonzero variance;
  * anti: every exact score negative, so that -1 sets the screen's floor;
  * minvar: winners whose var1_n sits on n^2 min_variance or within 2 var_margin(n) of it.
The keys are built from a chosen raw disparity: NoDuplicates keys for every family, and Consistency keys whose reverse
column gives odd sums, lands col1 on the border and outside the row, and puts |col - rev| at max_lr_diff and one past.
On the CPU: each family reaches its cases (counted), and the key builders round-trip through a numpy restatement of
the postfilter. On the GPU: uint8 float over every stack-size bucket and the screen's step-count edges, uint16,
double, a positive threshold, pitched input, ragged columns, 65535 rows and 32767 columns.
"""

import functools
import time

import numpy as np
import pytest

from libbicos_b200 import Config

F32 = np.float32
U = 2.0 ** -24
INVALID = -32768
THR = -2.0  # below every score: each evaluated pixel keeps d - best_x, so best_x is compared everywhere
MASK = {np.uint8: 0xFF, np.uint16: 0xFFFF}

# uint8 float, the screened path: every stack-size bucket (exact, just above, n = 2, 3 mod 4) and the step counts at
# the screen's limits: 1, 2, 3, 5, 7, 20, 29, 31, 32 (bit 31 of the survivor mask), 33 (above MAX_BOUNDED), 41, 201
NS_U8 = [2, 3, 4, 5, 8, 9, 10, 13, 16, 17, 18, 31, 32, 33, 34, 47, 64, 65]
STEPS_U8 = [2.5, 2.0, 1.0, 0.5, 0.3, 0.1, 0.07, 0.066, 0.0645, 0.0625, 0.049, 0.01]


def steps(step):
    """the x values of the reference's `for (float x = -1; x <= 1; x += step)`"""
    xs, x = [], F32(-1.0)
    while x <= F32(1.0):
        xs.append(x)
        x = F32(x + F32(step))
    return np.array(xs, F32)


def screen_margin(n):
    return (4 * n + 40) * U


def var_margin(n):
    return (n + 5) * U


def interp(y0, y1, y2, x, mask=None):
    """the kernel's rounded values ((a x) x + b x) + c in float32, round half even; wrapped to the input type by
    `mask`, unwrapped without it. x broadcasts over the last (pixel) axis."""
    a = F32(0.5) * (y0 - 2 * y1 + y2).astype(F32)
    b = F32(0.5) * (y2 - y0).astype(F32)
    x = np.asarray(x, F32)
    v = np.rint(((a * x) * x + b * x) + y1.astype(F32)).astype(np.int64)
    return v if mask is None else v & mask


def exact_scores(L, Y, xs, mask):
    """per step and pixel [steps, P]: the exact correlation of the wrapped values (NaN where a variance is 0), their
    var1_n = n S v^2 - (S v)^2, and whether an unwrapped value leaves [0, mask]"""
    n = L.shape[0]
    L = L.astype(np.int64)
    sl = L.sum(0)
    var0 = n * (L * L).sum(0) - sl * sl
    rho, var1, out = [], [], []
    for x in xs:
        v = interp(*Y, x)
        out.append(((v < 0) | (v > mask)).any(0))
        v &= mask
        sv = v.sum(0)
        v1 = n * (v * v).sum(0) - sv * sv
        cov = n * (L * v).sum(0) - sl * sv
        with np.errstate(divide="ignore", invalid="ignore"):
            rho.append(cov / np.sqrt(var0.astype(np.float64) * v1.astype(np.float64)))
        var1.append(v1)
    return np.stack(rho), np.stack(var1), np.stack(out)


def candidates(rho, n):
    """steps within screen_margin(n) of max(-1, best exact score) [steps, P] (NaN steps are never candidates)"""
    best = np.maximum(np.nanmax(np.where(np.isnan(rho), -np.inf, rho), axis=0), -1.0)
    return np.nan_to_num(rho, nan=-np.inf) >= best - screen_margin(n)


# ----------------------------------------------------------------------------------------------- families --
def _smooth_triples(rng, n, P, hi, spread):
    """triples whose parabolas stay well inside [0, hi]"""
    lo_c, hi_c = 2 * spread, hi - 2 * spread
    c = rng.integers(lo_c, hi_c + 1, size=(n, P))
    return np.stack([c + rng.integers(-spread, spread + 1, size=(n, P)), c,
                     c + rng.integers(-spread, spread + 1, size=(n, P))]).astype(np.int64)


def _noise(rng, L, hi, p=0.3):
    """+-1 on a few images of a share p of the pixels"""
    n, P = L.shape
    hit = (rng.random((n, P)) < 2.0 / n) & (rng.random((1, P)) < p)
    return np.clip(L + hit * rng.choice([-1, 1], size=(n, P)), 0, hi)


def fam_interp(rng, n, P, hi, xs, midpoint_share=0.3):
    """left = the rounded interpolation at a grid step (the first and last among them), a midpoint of two grid steps
    or a random x, with +-1 noise on some. Half the triples vary slowly (spread 1 to 3): neighbouring steps round to
    the same values there, which makes ties and pixels with many candidates."""
    spread = np.where(rng.random(P) < 0.5, max(2, hi // 10), rng.integers(1, 4, size=P))
    Y = _smooth_triples(rng, n, P, hi, spread)
    k = rng.integers(0, len(xs), size=P)
    k[: P // 16] = 0
    k[P // 16: P // 8] = len(xs) - 1
    x = xs[k].copy()
    kind = rng.random(P)
    if len(xs) > 1:
        mid = kind < midpoint_share
        km = np.minimum(k, len(xs) - 2)
        x[mid] = ((xs[km].astype(np.float64) + xs[km + 1]) / 2).astype(F32)[mid]
    rnd = kind > 0.85
    x[rnd] = rng.uniform(-1, 1, size=int(rnd.sum())).astype(F32)
    x[: P // 8] = xs[k[: P // 8]]  # the first and last grid step exactly
    L = interp(*Y, x[None, :], hi)
    L[:, P // 8:] = _noise(rng, L[:, P // 8:], hi)
    return L, Y


@functools.lru_cache(maxsize=None)
def edge_pools(hi):
    """Triples near the top of [0, hi] by the kind of their parabola's maximum on [-1, 1] (A = y0 - 2 y1 + y2 < 0,
    B = y2 - y0): "over" leaves the range by 1/2 or more, "half" by less than 1/2 (flagged, rounds back in range),
    "touch" reaches hi exactly at an inner vertex (t1 = 0), "end" has its vertex exactly at x = +-1 (t2 = 0, |B| = 2|A|).
    With 8 |A| eps = 8 |A| (y1 - hi) + B^2 the overshoot eps is exact in integers. Mirror (hi - y) for the bottom."""
    rng = np.random.default_rng(hi)
    if hi == 0xFF:
        y1, y0, y2 = np.meshgrid(np.arange(243, 256), np.arange(183, 256), np.arange(183, 256), indexing="ij")
        y0, y1, y2 = (v.ravel().astype(np.int64) for v in (y0, y1, y2))
    else:
        m = 100_000
        y1 = rng.integers(hi - 40, hi + 1, size=m)
        y0 = rng.integers(hi - 600, hi + 1, size=m)
        y2 = rng.integers(hi - 600, hi + 1, size=m)
    A, B = y0 - 2 * y1 + y2, y2 - y0
    inner = (A < 0) & (np.abs(B) < -2 * A)
    e8 = -8 * A * (y1 - hi) + B * B  # 8 |A| eps
    pools = {
        "over": inner & (e8 >= -4 * A),
        "half": inner & (e8 > 0) & (e8 < -4 * A),
        "touch": inner & (e8 == 0),
        "end": (A < 0) & (np.abs(B) == -2 * A),
    }
    return {k: np.stack([y0[v], y1[v], y2[v]]) for k, v in pools.items()}


def fam_wrap(rng, n, P, hi, xs):
    """Each pixel takes one kind of edge triple (top or bottom of the range) for most of its images; the left stack is
    the wrapped interpolation at the grid step where the most images leave the range (a random step if none does)."""
    pools = edge_pools(hi)
    kinds = list(pools)
    Y = _smooth_triples(rng, n, P, hi, max(2, hi // 10))
    kind = np.arange(P) % len(kinds)
    for i, name in enumerate(kinds):
        pool = pools[name]
        assert pool.shape[1] > 0, name
        cols = np.nonzero(kind == i)[0]
        take = rng.random((n, cols.size)) < 0.75
        pick = pool[:, rng.integers(0, pool.shape[1], size=(n, cols.size))]  # [3, n, c]
        bottom = rng.random(cols.size) < 0.5
        pick = np.where(bottom[None, None, :], hi - pick, pick)
        flip = rng.random((n, cols.size)) < 0.5  # the vertex on either side
        pick = np.where(flip[None], pick[::-1], pick)
        Y[:, :, cols] = np.where(take[None], pick, Y[:, :, cols])
    outs = np.stack([((interp(*Y, x) < 0) | (interp(*Y, x) > hi)).sum(0) for x in xs])  # [steps, P]
    k = np.where(outs.max(0) > 0, outs.argmax(0), rng.integers(0, len(xs), size=P))
    L = interp(*Y, xs[k][None, :], hi)
    return L, Y


def fam_flat(rng, n, P, hi, xs):
    """nearly constant triples (tiny var_q: no bound), constant triples (var1_n = 0 at every step: NaN), a constant left
    stack and a left stack of the smallest nonzero variance (one image off by one)"""
    q = P // 4
    Y = _smooth_triples(rng, n, P, hi, max(2, hi // 10))
    base = rng.integers(1, hi, size=(1, P))
    near = base + (rng.random((3, n, P)) < 0.2)
    Y[:, :, :q] = near[:, :, :q]
    Y[:, :, q:2 * q] = base[None, :, q:2 * q]
    L = rng.integers(0, hi + 1, size=(n, P))
    L[:, :q] = interp(*Y[:, :, :q], xs[rng.integers(0, len(xs), size=q)][None, :], hi)
    L[:, 2 * q:3 * q] = base[:, 2 * q:3 * q]
    L[:, 3 * q:] = base[:, 3 * q:]
    L[rng.integers(0, n, size=P - 3 * q), np.arange(3 * q, P)] += 1
    return L, Y


def fam_anti(rng, n, P, hi, xs):
    """left = the mirrored interpolation (hi - v) with noise, kept where every finite exact score is negative"""
    keepL, keepY = [], []
    for _ in range(50):
        if sum(v.shape[1] for v in keepL) >= P:
            break
        Y = _smooth_triples(rng, n, 4 * P, hi, max(2, hi // 10))
        L = _noise(rng, hi - interp(*Y, rng.choice(xs, size=4 * P)[None, :], hi), hi, p=0.5)
        rho, _, _ = exact_scores(L, Y, xs, hi)
        ok = (np.nan_to_num(rho, nan=-1.0) < 0).all(0) & np.isfinite(rho).any(0)
        keepL.append(L[:, ok])
        keepY.append(Y[:, :, ok])
    return np.concatenate(keepL, 1)[:, :P], np.concatenate(keepY, 2)[:, :, :P]


def fam_minvar(oracle, rng, n, P, hi, xs, step, dtype):
    """Pixels whose likely winner (the left stack is its interpolation, stretched) has var1_n exactly V0 (the images
    of one base pixel permuted) or within 2 var_margin(n) V0 of it (one image's triple shifted by +-1). Returns
    (L, Y, min_variance) with n^2 min_variance on V0."""
    k = int(rng.integers(0, len(xs)))
    spread = max(2, hi // 8)
    for _ in range(1000):
        Y0 = _smooth_triples(rng, n, 1, hi, spread)[:, :, 0]  # [3, n]
        Y0 = np.clip(Y0 - int(Y0[1].mean()) + (hi + 1) // 2, spread, hi - spread)  # centred: room for the stretch
        Y0[1] = np.clip(Y0[1], hi // 4, hi - hi // 4)
        v = interp(*Y0[:, :, None], xs[k])[:, 0]
        if v.min() >= 0 and v.max() <= hi and len(set(v.tolist())) > 1:
            break
    V0 = int(n * (v * v).sum() - v.sum() ** 2)
    window = 2 * var_margin(n) * V0
    variants = [Y0]
    for t in range(n):
        for dlt in (-1, 1):
            Yv = Y0.copy()
            Yv[:, t] += dlt
            vv = interp(*Yv[:, :, None], xs[k])[:, 0]
            if Yv.min() < 0 or Yv.max() > hi:
                continue
            if abs(int(n * (vv * vv).sum() - vv.sum() ** 2) - V0) <= window:
                variants.append(Yv)
    Y = np.empty((3, n, P), np.int64)
    for p in range(P):
        base = variants[p % len(variants)] if p % 2 else Y0  # half exactly on V0
        Y[:, :, p] = base[:, rng.permutation(n)]
    vk = interp(*Y, xs[k])
    m = vk.mean(0, keepdims=True)
    L = np.clip(np.rint(m + 1.5 * (vk - m)), 0, hi).astype(np.int64)  # var0 well above the boundary
    # min_variance a few float32 ulps around V0 / n^2: the one at which the oracle's float test keeps that step as the
    # winner in about half of the pixels, so that the float rounding decides
    base = np.array([np.float64(V0) / n / n], F32).view(np.int32)[0]
    best = None
    for j in range(-16, 17):
        mv = float(np.array([base + j], np.int32).view(F32)[0])
        bx, _ = _float_winners(oracle, L, Y, step, dtype, mv)
        share = float(np.mean(bx == xs[k]))
        if best is None or abs(share - 0.5) < best[0]:
            best = (abs(share - 0.5), mv)
    return L, Y, best[1]


def _float_winners(oracles, L, Y, step, dtype, mv=None):
    """the oracle's chosen x and score per pixel: each pixel alone in a row of three columns, d = 0"""
    n, P = L.shape
    left = np.zeros((n, P, 3), dtype)
    right = np.stack([Y[0], Y[1], Y[2]], axis=-1).astype(dtype)
    left[:, :, 1] = L
    raw = np.full((P, 3), INVALID, np.int16)
    raw[:, 1] = 0
    disp, corr = oracles.port.agree(raw, left, right, THR, step, mv)
    return -disp[:, 1], corr[:, 1]


def mine(oracles, rng, n, step, hi, dtype, want=(64, 128, 128), budget_s=0.5, batch=2048):
    """Interp pixels (half of them at midpoints) whose float winner is not the exact argmax, with three or more, and
    with exactly two candidates, up to `want` of each, within a CPU time budget. Returns (L, Y, counts)."""
    xs = steps(step)
    got = [[], [], []]
    t0 = time.process_time()
    while True:
        L, Y = fam_interp(rng, n, batch, hi, xs, midpoint_share=0.5)
        rho, _, _ = exact_scores(L, Y, xs, hi)
        cand = candidates(rho, n).sum(0)
        bx, _ = _float_winners(oracles, L, Y, step, dtype)
        finite = np.isfinite(rho).any(0)
        arg = np.nanargmax(np.where(np.isnan(rho), -np.inf, rho), axis=0)
        classes = [finite & (bx != xs[arg]), cand >= 3, cand == 2]
        for c, sel in enumerate(classes):
            have = sum(g.shape[1] for g, _ in got[c])
            idx = np.nonzero(sel & ~np.any(classes[:c], axis=0) if c else sel)[0][: max(0, want[c] - have)]
            if idx.size:
                got[c].append((L[:, idx], Y[:, :, idx]))
        full = all(sum(g.shape[1] for g, _ in got[c]) >= want[c] for c in range(3))
        if full or time.process_time() - t0 > budget_s:
            break
    parts = [p for g in got for p in g]
    counts = [sum(g.shape[1] for g, _ in got[c]) for c in range(3)]
    if not parts:
        return np.zeros((n, 0), np.int64), np.zeros((3, n, 0), np.int64), counts
    return np.concatenate([p[0] for p in parts], 1), np.concatenate([p[1] for p in parts], 2), counts


FAMILIES = ("interp", "wrap", "mined", "flat", "anti", "minvar")


@functools.lru_cache(maxsize=None)
def _families_cached(oracle, n, step, dtype_name, sizes, budget_s):
    dtype = np.dtype(dtype_name).type
    hi = MASK[dtype]
    xs = steps(step)
    rng = np.random.default_rng([n, len(xs), hi])
    fam = {}
    fam["interp"] = fam_interp(rng, n, sizes[0], hi, xs)
    fam["wrap"] = fam_wrap(rng, n, sizes[1], hi, xs)
    L, Y, counts = mine(oracle, rng, n, step, hi, dtype, budget_s=budget_s)
    fam["mined"] = (L, Y)
    fam["flat"] = fam_flat(rng, n, sizes[2], hi, xs)
    fam["anti"] = fam_anti(rng, n, sizes[3], hi, xs)
    L, Y, mv = fam_minvar(oracle, rng, n, sizes[4], hi, xs, step, dtype)
    fam["minvar"] = (L, Y)
    return fam, mv, counts


def families(oracles, n, step, dtype, sizes=(256, 192, 64, 64, 96), budget_s=0.5):
    """{family: (L [n, P], Y [3, n, P])}, the scene's min_variance edge, and the mined counts"""
    return _families_cached(oracles, n, step, np.dtype(dtype).name, tuple(sizes), budget_s)


# ------------------------------------------------------------------------------------------------- layout --
def layout(fam, dtype, seed, groups_per_row=43, extra=2, min_rows=1):
    """Lay the pixels out as stacks [n, rows, cols] and a raw disparity [rows, cols].

    Each family pixel gets a group of three right columns holding its triple; the three left pixels of a left group
    all take the centre column of the right group a random permutation gives them (d from -cols to cols), one of them
    the family pixel and two others refined against the same triple at random x. In each row one of those fillers
    takes col1 = 0 and one col1 = cols - 1 (the integer NXC branch), the `extra` columns beyond the groups take random
    columns, and 3 % of the fillers are invalid. Returns left, right and raw."""
    rng = np.random.default_rng(seed)
    hi = MASK[dtype]
    L = np.concatenate([fam[k][0] for k in fam], 1)
    Y = np.concatenate([fam[k][1] for k in fam], 2)
    n, P = L.shape
    gpr = groups_per_row
    rows = max(min_rows, -(-P // gpr))
    cols = 3 * gpr + extra
    G = rows * gpr
    # pad with interp pixels
    if G > P:
        Lp, Yp = fam_interp(rng, n, G - P, hi, steps(0.1))
        L, Y = np.concatenate([L, Lp], 1), np.concatenate([Y, Yp], 2)
    left = rng.integers(0, hi + 1, size=(n, rows, cols)).astype(np.int64)
    right = rng.integers(0, hi + 1, size=(n, rows, cols)).astype(np.int64)
    raw = np.zeros((rows, cols), np.int64)
    filler = np.zeros((rows, cols), bool)
    r_of = np.repeat(np.arange(rows), gpr)
    j_of = np.tile(np.arange(gpr), rows)
    perm = np.stack([rng.permutation(gpr) for _ in range(rows)])
    g_of = perm[r_of, j_of]
    for k in range(3):
        right[:, r_of, 3 * g_of + k] = Y[k]
    slot = rng.integers(0, 3, size=G)
    xf = rng.uniform(-1, 1, size=(3, G)).astype(F32)
    for s in range(3):
        c = 3 * j_of + s
        own = slot == s
        Lf = _noise(rng, interp(*Y, xf[s][None, :], hi), hi)
        left[:, r_of, c] = np.where(own[None, :], L, Lf)
        raw[r_of, c] = c - (3 * g_of + 1)
        filler[r_of[~own], c[~own]] = True
    col = np.arange(cols)
    for r in range(rows):
        f = np.nonzero(filler[r, : 3 * gpr])[0]
        b = rng.choice(f, size=2, replace=False)
        raw[r, b[0]] = b[0] - 0
        raw[r, b[1]] = b[1] - (cols - 1)
    raw[:, 3 * gpr:] = col[3 * gpr:] - rng.integers(0, cols, size=(rows, extra))
    filler[:, 3 * gpr:] = True
    invalid = filler & (rng.random((rows, cols)) < 0.03)
    raw[invalid] = INVALID
    return left.astype(dtype), right.astype(dtype), raw.astype(np.int16)


def nodupes_keys(raw, rng):
    """fwd_first = cost << 16 | col1 and fwd_last = cost' << 16 | (65535 - col1) with random costs; a mismatching
    fwd_last where raw is invalid"""
    rows, cols = raw.shape
    col = np.arange(cols)[None, :]
    valid = raw != INVALID
    col1 = np.where(valid, col - raw.astype(np.int64), rng.integers(0, cols, size=raw.shape))
    low = 65535 - col1
    low = np.where(valid, low, low ^ rng.integers(1, 65536, size=raw.shape))
    ff = rng.integers(0, 65536, size=raw.shape).astype(np.uint32) << 16 | col1.astype(np.uint32)
    fl = rng.integers(0, 65536, size=raw.shape).astype(np.uint32) << 16 | low.astype(np.uint32)
    return ff, fl


def postfilter(ff, fl, rf, rl, consistency, no_dupes, max_lr):
    """numpy restatement of refine_kernel's postfilter (bicos.hpp:95-110) -> raw int16"""
    rows, cols = ff.shape
    r = np.arange(rows)[:, None]
    col = np.arange(cols)[None, :]
    best = (ff & 0xFFFF).astype(np.int64)
    valid = np.ones((rows, cols), bool)
    if not consistency or no_dupes:
        valid &= (fl & 0xFFFF).astype(np.int64) == 65535 - best
    if consistency:
        rev = (rf[r, best] & 0xFFFF).astype(np.int64)
        if no_dupes:
            valid &= (rl[r, best] & 0xFFFF).astype(np.int64) == 65535 - rev
        valid &= np.abs(col - rev) <= max_lr
        d = (col + rev) // 2 - best
    else:
        d = col - best
    return np.where(valid, d, INVALID).astype(np.int16)


def consistency_keys(rows, cols, max_lr, no_dupes, seed):
    """Keys of a Consistency config: left column c takes right column b (a permutation per row), whose reverse key
    holds rev = c + delta, delta cycling through 0, +-1, +-2, +-max_lr, +-(max_lr + 1) and random values (odd and even
    sums, |col - rev| at max_lr and one past). The pixels taking b = 0 and b = cols - 1 cycle through deltas that put
    col1 = b - floor(delta / 2) on the border and outside the row. A few fwd_last / rev_last keys mismatch."""
    rng = np.random.default_rng(seed)
    deltas = np.array([0, 1, -1, 2, -2, 3, -3, max_lr, -max_lr, max_lr + 1, -(max_lr + 1), max_lr - 1, 1 - max_lr])
    b = np.stack([rng.permutation(cols) for _ in range(rows)])
    delta = np.where(rng.random((rows, cols)) < 0.8, deltas[rng.integers(0, deltas.size, (rows, cols))],
                     rng.integers(-3 * max_lr - 3, 3 * max_lr + 4, (rows, cols)))
    r = np.arange(rows)[:, None]
    c = np.broadcast_to(np.arange(cols)[None, :], (rows, cols))
    edge = np.array([0, 1, -1, 2, -2, 3])
    e0, e1 = np.argmax(b == 0, axis=1), np.argmax(b == cols - 1, axis=1)
    delta[np.arange(rows), e0] = edge[np.arange(rows) % edge.size]
    delta[np.arange(rows), e1] = edge[(np.arange(rows) + 3) % edge.size]
    rev = np.maximum(c + delta, 0)
    ff = rng.integers(0, 65536, size=(rows, cols)).astype(np.uint32) << 16 | b.astype(np.uint32)
    fl = rng.integers(0, 65536, size=(rows, cols)).astype(np.uint32) << 16 | (65535 - b).astype(np.uint32)
    rf = np.zeros((rows, cols), np.uint32)
    rl = np.zeros((rows, cols), np.uint32)
    rf[r, b] = rng.integers(0, 65536, size=(rows, cols)).astype(np.uint32) << 16 | rev.astype(np.uint32)
    rl[r, b] = rng.integers(0, 65536, size=(rows, cols)).astype(np.uint32) << 16 | (65535 - rev).astype(np.uint32)
    bad = rng.random((rows, cols)) < 0.03
    fl[bad] ^= 1
    bad = rng.random((rows, cols)) < 0.03
    rl[bad] ^= 2
    return ff, fl, rf, rl, rev, b


def consistency_scene(n, rows, cols, raw, dtype, seed):
    """a smooth right stack; each valid interior left pixel is its rounded interpolation at col1 and a random x"""
    rng = np.random.default_rng(seed)
    hi = MASK[dtype]
    right = np.clip(hi // 2 + np.cumsum(rng.integers(-hi // 12, hi // 12 + 1, size=(n, rows, cols)), axis=2), 0, hi)
    left = rng.integers(0, hi + 1, size=(n, rows, cols)).astype(np.int64)
    rr, cc = np.nonzero(raw != INVALID)
    c1 = cc - raw[rr, cc].astype(np.int64)
    inner = (c1 > 0) & (c1 < cols - 1)
    rr, cc, c1 = rr[inner], cc[inner], c1[inner]
    Y = np.stack([right[:, rr, c1 - 1], right[:, rr, c1], right[:, rr, c1 + 1]])
    x = rng.uniform(-1, 1, size=rr.size).astype(F32)
    left[:, rr, cc] = _noise(rng, interp(*Y, x[None, :], hi), hi)
    return left.astype(dtype), right.astype(dtype)


# ------------------------------------------------------------------------------------------------ CPU side --
def test_steps_hit_the_screen_limits():
    counts = {s: len(steps(s)) for s in STEPS_U8}
    assert counts == {2.5: 1, 2.0: 2, 1.0: 3, 0.5: 5, 0.3: 7, 0.1: 20, 0.07: 29, 0.066: 31, 0.0645: 32, 0.0625: 33,
                      0.049: 41, 0.01: 201}


def test_edge_pools_are_exact():
    """the kinds of edge triple agree with the kernel's float wrap test (t1, t2) and with the rounded values"""
    for hi in (0xFF, 0xFFFF):
        for name, Y in edge_pools(hi).items():
            assert Y.shape[1] > 0, (hi, name)
            y0, y1, y2 = (v.astype(F32) for v in Y)
            a, b = F32(0.5) * (y0 - 2 * y1 + y2), F32(0.5) * (y2 - y0)
            t2 = 4 * a.astype(np.float64) ** 2 - b.astype(np.float64) ** 2
            t1 = b.astype(np.float64) ** 2 - 510 * np.abs(a) - 4 * a * (y1 - 127.5) if hi == 0xFF else None
            if name == "end":
                assert (t2 == 0).all()
            else:
                assert (t2 > 0).all()
            if t1 is not None:
                assert {"over": (t1 > 0).all(), "half": (t1 > 0).all(), "touch": (t1 == 0).all(),
                        "end": True}[name], name
            vmax = np.stack([interp(*Y, x) for x in np.linspace(-1, 1, 401, dtype=F32)]).max(0)
            if name == "half" and hi == 0xFF:  # (near 65535 the float32 interpolation errs by up to 2^-8)
                assert (vmax <= hi).all(), "an overshoot below 1/2 rounds back into the range"
            if name == "over":
                assert (vmax > hi).mean() > 0.9


@pytest.mark.parametrize("n,step", [(33, 0.1), (33, 0.0645), (9, 0.066), (64, 0.049)])
def test_families_reach_their_cases(oracles, n, step):
    """Counted on uint8 scenes: wrap-flagged pixels whose float winner is a wrapped step (and whose bound at the winner
    is below the floor: a screen that bounded them would drop the winner), t1 == 0 pixels, exact ties, two- and
    three-or-more-candidate pixels, float winners that are not the exact argmax, near-min-variance winners, border
    pixels, and winners at step 31 of the 32-step grid."""
    import importlib.util
    import os

    hi, xs = 0xFF, steps(step)
    fam, mv, mined = families(oracles, n, step, np.uint8, budget_s=3.0)
    spec = importlib.util.spec_from_file_location(
        "refine_candidates", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "refine_candidates.py"))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    counts = {}

    L, Y = fam["wrap"]
    rho, _, out = exact_scores(L, Y, xs, hi)
    bx, best = _float_winners(oracles, L, Y, step, np.uint8)
    kw = np.argmax(xs[:, None] == bx[None, :], axis=0)
    wraps, ub, _ = tool.kernel_bound(L, *Y, xs)
    P = L.shape[1]
    wrapped_winner = wraps & out[kw, np.arange(P)] & np.isfinite(best)
    counts["wrap_winner"] = int(wrapped_winner.sum())
    floor = np.maximum(np.nanmax(np.where(np.isnan(rho), -np.inf, rho), 0), -1) - screen_margin(n)
    counts["wrap_winner_below_bound"] = int((wrapped_winner & (ub[kw, np.arange(P)] < floor)).sum())
    y0, y1, y2 = (v.astype(np.float64) for v in Y)
    a, b = 0.5 * (y0 - 2 * y1 + y2), 0.5 * (y2 - y0)
    t1 = b * b - 510 * np.abs(a) - 4 * a * (y1 - 127.5)
    t2 = 4 * a * a - b * b
    counts["t1_zero"] = int(((t1 == 0) & (t2 > 0)).any(0).sum())

    allL = np.concatenate([fam[k][0] for k in ("interp", "mined", "anti")], 1)
    allY = np.concatenate([fam[k][1] for k in ("interp", "mined", "anti")], 2)
    rho, _, _ = exact_scores(allL, allY, xs, hi)
    r = np.where(np.isnan(rho), -np.inf, rho)
    top = r.max(0)
    counts["exact_ties"] = int((((r == top) & np.isfinite(top)).sum(0) >= 2).sum())
    cand = candidates(rho, n).sum(0)
    counts["two_candidates"] = int((cand == 2).sum())
    counts["three_or_more"] = int((cand >= 3).sum())
    bx, _ = _float_winners(oracles, allL, allY, step, np.uint8)
    counts["float_not_exact_argmax"] = int((np.isfinite(top) & (bx != xs[np.argmax(r, 0)])).sum())

    L, Y = fam["anti"]
    rho, _, _ = exact_scores(L, Y, xs, hi)
    counts["anti"] = int((np.nan_to_num(rho, nan=-1) < 0).all(0).sum())

    L, Y = fam["minvar"]
    _, var1, _ = exact_scores(L, Y, xs, hi)
    bx, _ = _float_winners(oracles, L, Y, step, np.uint8, mv)
    kw = np.argmax(xs[:, None] == bx[None, :], axis=0)
    mvn = np.float64(F32(F32(mv) * F32(n))) * n
    near = np.abs(var1 - mvn) <= 2 * var_margin(n) * mvn
    counts["near_minvar_winner"] = int(near[kw, np.arange(L.shape[1])].sum())
    counts["near_minvar_any"] = int(near.any(0).sum())

    left, right, raw = layout(fam, np.uint8, seed=n)
    c1 = np.arange(raw.shape[1])[None, :] - raw.astype(np.int64)
    valid = raw != INVALID
    counts["border"] = int((valid & ((c1 == 0) | (c1 == raw.shape[1] - 1))).sum())
    counts["invalid"] = int((~valid).sum())
    print(n, step, counts, "mined", mined)

    assert counts["wrap_winner"] >= 20
    assert counts["wrap_winner_below_bound"] >= 1
    assert counts["t1_zero"] >= 20
    assert counts["exact_ties"] >= 10
    assert counts["two_candidates"] >= 20 and counts["three_or_more"] >= 20
    assert counts["float_not_exact_argmax"] >= 1
    assert counts["anti"] == fam["anti"][0].shape[1]
    assert counts["near_minvar_winner"] >= 10
    assert counts["border"] >= raw.shape[0] and counts["invalid"] >= 1
    if len(xs) == 32:
        L, Y = fam["interp"]
        bx, _ = _float_winners(oracles, L, Y, step, np.uint8)
        assert (bx == xs[31]).sum() >= 8, "winners at bit 31 of the survivor mask"


def test_nodupes_keys_round_trip(oracles):
    fam, _, _ = families(oracles, 9, 0.1, np.uint8, sizes=(64, 16, 16, 16, 16), budget_s=0.1)
    _, _, raw = layout(fam, np.uint8, seed=3)
    ff, fl = nodupes_keys(raw, np.random.default_rng(0))
    assert (ff >> 16).any() and (fl >> 16).any(), "random cost bits above the column"
    assert np.array_equal(postfilter(ff, fl, None, None, False, False, 1), raw)
    for no_dupes in (False, True):
        ff, fl, rf, rl, rev, b = consistency_keys(24, 131, 3, no_dupes, seed=1)
        got = postfilter(ff, fl, rf, rl, True, no_dupes, 3)
        c = np.arange(131)[None, :]
        want = np.where(np.abs(c - rev) <= 3, (c + rev) // 2 - b, INVALID)
        ok = np.ones(b.shape, bool)
        if no_dupes:  # Consistency checks fwd_last only with no_dupes (search_flags: NODUPES | CONSISTENCY)
            ok &= (fl & 0xFFFF) == 65535 - b
            ok &= np.take_along_axis(rl & 0xFFFF, b, 1) == 65535 - np.take_along_axis(rf & 0xFFFF, b, 1)
        want = np.where(ok, want, INVALID)
        assert np.array_equal(got, want.astype(np.int16))


def test_consistency_keys_reach_their_edges():
    rows, cols, max_lr = 24, 131, 3
    ff, fl, rf, rl, rev, b = consistency_keys(rows, cols, max_lr, True, seed=1)
    c = np.arange(cols)[None, :]
    raw = postfilter(ff, fl, rf, rl, True, True, max_lr)
    valid = raw != INVALID
    c1 = c - raw.astype(np.int64)
    assert (valid & ((c + rev) % 2 == 1)).sum() > 100, "odd sums"
    assert (valid & (c1 == 0)).sum() >= 3 and (valid & (c1 == cols - 1)).sum() >= 3
    assert (valid & ((c1 < 0) | (c1 >= cols))).sum() >= 3, "col1 outside the row"
    assert (valid & (np.abs(c - rev) == max_lr)).sum() > 20
    assert (np.abs(c - rev) == max_lr + 1).sum() > 20 and not (valid & (np.abs(c - rev) > max_lr)).any()


# ------------------------------------------------------------------------------------------------ GPU side --
def _cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _keys(*keys):
    return tuple(None if k is None else _cuda(k.view(np.int32)) for k in keys)


def _stacks(left, right, pad):
    """device stacks; with `pad`, [:, :, :cols] views of planes `pad` columns wider"""
    if not pad:
        return _cuda(left), _cuda(right)
    n, rows, cols = left.shape

    def wide(a):
        w = np.zeros((n, rows, cols + pad), a.dtype)
        w[:, :, :cols] = a
        w[:, :, cols:] = a[:, :, :pad] if pad <= cols else 0
        return _cuda(w)[:, :, :cols]

    return wide(left), wide(right)


def _refine_and_compare(handle, oracles, left, right, raw, keys, cfg, pad=0):
    l, r = _stacks(left, right, pad)
    disp, corr, got_raw = handle.refine(l, r, cfg, _keys(*keys))
    want_d, want_c = oracles.port.agree(raw, left, right, cfg.nxcorr_threshold, cfg.subpixel_step, cfg.min_variance,
                                        double=cfg.double)
    got_raw, got_d, got_c = got_raw.cpu().numpy(), disp.cpu().numpy(), corr.cpu().numpy()
    assert np.array_equal(got_raw, raw), f"{(got_raw != raw).sum()} raw disparities differ"
    bad_c = ~((got_c == want_c) | (np.isnan(got_c) & np.isnan(want_c)))
    bad_d = ~((got_d == want_d) | (np.isnan(got_d) & np.isnan(want_d)))
    where = np.argwhere(bad_c | bad_d)[:3].tolist()
    assert not bad_c.any(), f"{bad_c.sum()} corrmap cells differ, first at {where}"
    assert not bad_d.any(), f"{bad_d.sum()} disparities differ, first at {where}"
    return want_c


def _run(handle, oracles, n, step, dtype, double, thresholds=(THR,), pad=0, sizes=(256, 192, 64, 64, 96),
         budget_s=0.5, **lay):
    fam, mv, _ = families(oracles, n, step, dtype, sizes=sizes, budget_s=budget_s)
    left, right, raw = layout(fam, dtype, seed=n * 1000 + len(steps(step)), **lay)
    keys = nodupes_keys(raw, np.random.default_rng(n)) + (None, None)
    for thr in thresholds:
        for minvar in (None, mv):
            cfg = Config(nxcorr_threshold=thr, subpixel_step=step, min_variance=minvar, double=double)
            want_c = _refine_and_compare(handle, oracles, left, right, raw, keys, cfg, pad=pad)
            assert np.isfinite(want_c).mean() > 0.8


@pytest.mark.gpu
@pytest.mark.parametrize("step", STEPS_U8)
@pytest.mark.parametrize("n", NS_U8)
def test_u8_float(handle, oracles, n, step):
    _run(handle, oracles, n, step, np.uint8, False)


@pytest.mark.gpu
@pytest.mark.parametrize("double", [False, True])
@pytest.mark.parametrize("step", [2.0, 0.3, 0.0645, 0.0625, 0.01])
@pytest.mark.parametrize("n", [2, 5, 17, 34, 65])
def test_u16(handle, oracles, n, step, double):
    _run(handle, oracles, n, step, np.uint16, double, sizes=(128, 192, 32, 32, 64), budget_s=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("step", [1.0, 0.1, 0.0625])
@pytest.mark.parametrize("n", [3, 9, 33, 47])
def test_u8_double(handle, oracles, n, step):
    _run(handle, oracles, n, step, np.uint8, True, sizes=(128, 128, 32, 32, 64), budget_s=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,double", [(np.uint8, False), (np.uint16, False), (np.uint8, True)])
@pytest.mark.parametrize("n,step", [(9, 0.1), (33, 0.0645), (18, 0.5)])
def test_positive_threshold(handle, oracles, n, step, dtype, double):
    """0.9 and 0.999: part of the evaluated pixels drop to NaN"""
    _run(handle, oracles, n, step, dtype, double, thresholds=(0.9, 0.999), sizes=(128, 64, 32, 32, 32), budget_s=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_pitched_input(handle, oracles, dtype):
    _run(handle, oracles, 33, 0.1, dtype, False, pad=40, sizes=(128, 64, 32, 32, 32), budget_s=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("gpr,extra", [(40, 1), (85, 0), (1, 2), (170, 1)])  # 121, 255, 5 and 511 columns
def test_ragged_columns(handle, oracles, gpr, extra):
    _run(handle, oracles, 17, 0.066, np.uint8, False, groups_per_row=gpr, extra=extra, sizes=(128, 64, 32, 32, 32),
         budget_s=0.2)


@pytest.mark.gpu
def test_rows_at_the_grid_limit(handle, oracles):
    """65535 rows (the refine's grid.y limit) of 5 columns"""
    _run(handle, oracles, 9, 0.1, np.uint8, False, groups_per_row=1, extra=2, min_rows=65535,
         sizes=(128, 64, 32, 32, 32), budget_s=0.2)


@pytest.mark.gpu
def test_columns_at_the_int16_limit(handle, oracles):
    """32767 columns: disparities up to +-32766"""
    _run(handle, oracles, 9, 0.1, np.uint8, False, groups_per_row=10922, extra=1, sizes=(128, 64, 32, 32, 32),
         budget_s=0.2)


@pytest.mark.gpu
@pytest.mark.parametrize("no_dupes", [False, True])
@pytest.mark.parametrize("n,step,dtype,double", [(9, 0.1, np.uint8, False), (33, 0.0645, np.uint8, False),
                                                 (33, None, np.uint8, False), (17, 0.3, np.uint16, False),
                                                 (10, 0.1, np.uint8, True)])
def test_consistency(handle, oracles, n, step, dtype, double, no_dupes):
    rows, cols, max_lr = 24, 131, 3
    ff, fl, rf, rl, _, _ = consistency_keys(rows, cols, max_lr, no_dupes, seed=n)
    raw = postfilter(ff, fl, rf, rl, True, no_dupes, max_lr)
    left, right = consistency_scene(n, rows, cols, raw, dtype, seed=n)
    keys = (ff, fl if no_dupes else None, rf, rl if no_dupes else None)
    for thr in (THR, 0.9):
        cfg = Config(nxcorr_threshold=thr, subpixel_step=step, consistency=True, max_lr_diff=max_lr, no_dupes=no_dupes,
                     double=double)
        _refine_and_compare(handle, oracles, left, right, raw, keys, cfg)
