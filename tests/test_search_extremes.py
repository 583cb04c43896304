"""Every search kernel at its cost and width limits, against exact keys; the whole match on degenerate pixel stacks.

The other search tests draw descriptors far from the numeric edges the kernels are built around: costs near 16 K bits,
widths up to 9000 columns, and engines compared with each other. Here:
- reference_keys() states the four key arrays of include/bicos_b200.h exactly (numpy, descriptors drawn from a small
  pool, so a 32767-wide row costs O(W * P)); a CPU test checks it against a brute force.
- extreme pools (zero, all usable bits, complements, one bit flipped, single bits) and rows whose minimum cost is at or
  next to the maximum usable cost B = 32 K - free bits, or where every pair ties at B or at 0;
- a case table that reaches every kernel name the dispatch can produce (asserted with last_search_kernel()), every
  tensor-core kernel at 8192 columns, the popcount engine and the windowed kernel at 32767;
- whole matches on constant, monotone, alternating, affine and anti-correlated stacks against the oracle, and the
  integer-mode correlation against an exact rational evaluation of the NXC.
"""

import os
from dataclasses import dataclass
from decimal import Decimal, localcontext
from typing import Optional, Tuple

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config

FLAG_NODUPES, FLAG_CONSISTENCY = 1, 2
KEY_NONE = 0xFFFFFFFF
KS = (1, 2, 4, 8, 12, 16)
COL_LIMIT_MMA = 8192  # rows of up to COL_MAX + 1 pixels on the tensor-core engine (search_mma.cu)
COL_LIMIT = 32767


# ------------------------------------------------------------------------------------------------ exact keys --
def popcount_words(a: np.ndarray) -> np.ndarray:
    """Set bits of [..., K] uint32 descriptors -> [...] int64."""
    return np.bitwise_count(np.ascontiguousarray(a, dtype=np.uint32)).sum(axis=-1, dtype=np.int64)


def _window_argmin(query: np.ndarray, cand: np.ndarray, table: np.ndarray, lo: np.ndarray, hi: np.ndarray):
    """For each query position q: over candidate positions j in [lo[q], hi[q]] (inclusive, empty if lo > hi), the
    minimum of table[query[q], cand[j]], the first and the last j attaining it. Per pool value v: its first and last
    position in the window by searchsorted. -> (cost, first, last, empty) with cost = -1 where empty."""
    big = np.iinfo(np.int64).max
    w = len(query)
    best = np.full(w, big, dtype=np.int64)
    first = np.full(w, big, dtype=np.int64)
    last = np.full(w, -1, dtype=np.int64)
    for v in np.unique(cand):
        pos = np.flatnonzero(cand == v)
        a = np.searchsorted(pos, lo, "left")  # first position >= lo
        b = np.searchsorted(pos, hi, "right") - 1  # last position <= hi
        present = a <= b
        fa = pos[np.minimum(a, len(pos) - 1)]
        lb_ = pos[np.maximum(b, 0)]
        c = np.where(present, table[query, v], big)
        better = c < best
        tie = (c == best) & present
        first = np.where(better, fa, np.where(tie, np.minimum(first, fa), first))
        last = np.where(better, lb_, np.where(tie, np.maximum(last, lb_), last))
        best = np.minimum(best, c)
    empty = best == big
    return np.where(empty, -1, best), first, last, empty


def _keys(cost, col, empty, mirror=False):
    k = (cost.astype(np.uint64) << np.uint64(16)) | ((65535 - col) if mirror else col).astype(np.uint64)
    return np.where(empty, KEY_NONE, k).astype(np.uint32)


def reference_keys(idx0: np.ndarray, idx1: np.ndarray, pool: np.ndarray, flags: int,
                   drange: Optional[Tuple[int, int]] = None):
    """The key arrays bicos_b200_search (drange None) or bicos_b200_search_range fills, for descriptors
    pool[idx0] (left) and pool[idx1] (right), idx [rows, cols] into a pool [P, K] of uint32 words:
      fwd_first  cost << 16 | first right column of the minimum, per left pixel
      fwd_last   with NODUPES: cost << 16 | 65535 - last right column; ranged without NODUPES the mirror of fwd_first
      rev_first  with CONSISTENCY: the same per right column over the left row
      rev_last   with NODUPES | CONSISTENCY
    Ranged: only pairs with min <= i - j <= max; an empty window is KEY_NONE. Arrays a search does not fill are None."""
    rows, cols = idx0.shape
    table = popcount_words(pool[:, None, :] ^ pool[None, :, :])  # [P, P], symmetric
    x = np.arange(cols, dtype=np.int64)
    if drange is None:
        fwd_win = rev_win = (np.zeros(cols, np.int64), np.full(cols, cols - 1, np.int64))
    else:
        dmin, dmax = drange
        fwd_win = (np.maximum(x - dmax, 0), np.minimum(x - dmin, cols - 1))  # right columns of left pixel x
        rev_win = (np.maximum(x + dmin, 0), np.minimum(x + dmax, cols - 1))  # left columns of right pixel x
    nodupes, cons = bool(flags & FLAG_NODUPES), bool(flags & FLAG_CONSISTENCY)
    out = {"fwd_first": np.empty((rows, cols), np.uint32)}
    out["fwd_last"] = np.empty((rows, cols), np.uint32) if nodupes or drange is not None else None
    out["rev_first"] = np.empty((rows, cols), np.uint32) if cons else None
    out["rev_last"] = np.empty((rows, cols), np.uint32) if nodupes and cons else None
    for r in range(rows):
        cost, first, last, empty = _window_argmin(idx0[r], idx1[r], table, *fwd_win)
        out["fwd_first"][r] = _keys(cost, first, empty)
        if nodupes:
            out["fwd_last"][r] = _keys(cost, last, empty, mirror=True)
        elif drange is not None:
            out["fwd_last"][r] = _keys(cost, first, empty, mirror=True)
        if cons:
            cost, first, last, empty = _window_argmin(idx1[r], idx0[r], table, *rev_win)
            out["rev_first"][r] = _keys(cost, first, empty)
            if nodupes:
                out["rev_last"][r] = _keys(cost, last, empty, mirror=True)
    return out


def brute_keys(d0: np.ndarray, d1: np.ndarray, flags: int, drange=None):
    """The same keys from the full cost matrix of each row, one pixel at a time."""
    rows, cols, _ = d0.shape
    nodupes, cons = bool(flags & FLAG_NODUPES), bool(flags & FLAG_CONSISTENCY)
    i = np.arange(cols)[:, None]
    j = np.arange(cols)[None, :]
    inr = np.ones((cols, cols), bool) if drange is None else (i - j >= drange[0]) & (i - j <= drange[1])
    names = ("fwd_first", "fwd_last", "rev_first", "rev_last")
    out = {k: np.full((rows, cols), KEY_NONE, np.uint32) for k in names}

    def first_last(costs, mask):
        if not mask.any():
            return None
        c = np.where(mask, costs, 1 << 40)
        at = np.flatnonzero(c == c.min())
        return int(c.min()), int(at[0]), int(at[-1])

    for r in range(rows):
        cost = popcount_words(d0[r][:, None, :] ^ d1[r][None, :, :])  # [left, right]
        for c in range(cols):
            f = first_last(cost[c], inr[c])
            if f is not None:
                out["fwd_first"][r, c] = f[0] << 16 | f[1]
                out["fwd_last"][r, c] = f[0] << 16 | (65535 - (f[2] if nodupes else f[1]))
            b = first_last(cost[:, c], inr[:, c])
            if b is not None:
                out["rev_first"][r, c] = b[0] << 16 | b[1]
                out["rev_last"][r, c] = b[0] << 16 | (65535 - b[2])
    if not (nodupes or drange is not None):
        out["fwd_last"] = None
    if not cons:
        out["rev_first"] = out["rev_last"] = None
    elif not nodupes:
        out["rev_last"] = None
    return out


def _decode(key: int, last: bool) -> str:
    if key == KEY_NONE:
        return "KEY_NONE"
    col = key & 0xFFFF
    return f"cost {key >> 16} col {65535 - col if last else col}"


def assert_keys_equal(got: dict, want: dict, what: str = "") -> None:
    """Every key array exactly; on a difference, the first differing pixel with both keys decoded."""
    for name, w in want.items():
        g = got.get(name)
        if w is None:
            continue
        assert g is not None, f"{what}: {name} missing"
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            r, c = (int(v) for v in bad[0])
            last = name.endswith("_last")
            raise AssertionError(f"{what}: {name} differs at {len(bad)} pixels, first (row {r}, col {c}): "
                                 f"got {_decode(int(g[r, c]), last)}, want {_decode(int(w[r, c]), last)}")


# --------------------------------------------------------------------------------------------- extreme pools --
@dataclass
class Pool:
    """Descriptors [P, K] whose set bits lie in bits 0 .. B - 1, with the indices the row patterns need."""

    words: np.ndarray
    bits: int
    zero: int
    ones: int
    rand: list  # random values
    comp: dict  # index -> index of its complement within B (zero <-> ones, random <-> complement)
    flip: dict  # index -> index of the same value with one bit flipped
    single: list  # single-bit values


def _ones(k: int, bits: int) -> np.ndarray:
    w = np.zeros(k, np.uint32)
    for b in range(bits):
        w[b // 32] |= np.uint32(1 << (b % 32))
    return w


def make_pool(k: int, free_bits: int, seed: int, nrand: int = 3) -> Pool:
    """Zero and all-B-ones; random values and their complements within B; each of those with one bit flipped;
    single-bit values at bit 0, B - 1 and in between. B = 32 K - free_bits."""
    rng = np.random.default_rng(seed)
    bits = 32 * k - free_bits
    mask = _ones(k, bits)
    vals = [np.zeros(k, np.uint32), mask.copy()]
    comp = {0: 1, 1: 0}
    rand = []
    for _ in range(nrand):
        v = rng.integers(0, 2**32, size=k, dtype=np.uint64).astype(np.uint32) & mask
        rand.append(len(vals))
        comp[len(vals)], comp[len(vals) + 1] = len(vals) + 1, len(vals)
        vals += [v, ~v & mask]
    flip = {}
    for i in range(len(vals)):
        b = int(rng.integers(0, bits))
        w = vals[i].copy()
        w[b // 32] ^= np.uint32(1 << (b % 32))
        flip[i] = len(vals)
        vals.append(w)
    single = []
    for b in sorted({0, bits - 1, bits // 2, int(rng.integers(0, bits))}):
        w = np.zeros(k, np.uint32)
        w[b // 32] = np.uint32(1 << (b % 32))
        single.append(len(vals))
        vals.append(w)
    words = np.stack(vals).astype(np.uint32)
    assert not (words & ~mask).any()
    return Pool(words, bits, 0, 1, rand, comp, flip, single)


def min_columns(cols: int):
    """Columns for a planted unique minimum: the first, either side of the first tile edge, the last column of the
    tensor-core engine's widest row, and the row's last column (inside a ragged tile when cols % 128 != 0)."""
    return sorted({c for c in (0, 127, 128, 8191, cols - 1) if 0 <= c < cols})


def pattern_rows(pool: Pool, cols: int, rng) -> list:
    """(idx0, idx1) rows of extreme patterns:
    - every pair at cost B (zero against all ones, all ones against zero, a random value against its complement),
      or every pair at cost 0 (all ones against all ones: left popcount B);
    - a unique minimum of cost B - 1 at each min_columns() column, forward (left uniform) and reverse (right uniform);
    - random rows of pool values, and rows of single-bit values."""
    P = len(pool.words)
    full = lambda v: np.full(cols, v, np.int64)  # noqa: E731
    rows = [(full(pool.zero), full(pool.ones)), (full(pool.ones), full(pool.zero)), (full(pool.ones), full(pool.ones)),
            (full(pool.rand[0]), full(pool.comp[pool.rand[0]]))]
    for t, c in enumerate(min_columns(cols)):
        v = pool.zero if t % 2 == 0 else pool.rand[t % len(pool.rand)]
        cv = pool.comp[v]
        right = full(cv)
        right[c] = pool.flip[cv]  # ham(v, flip(comp v)) = B - 1, every other column B
        rows.append((full(v), right))
        v = pool.rand[(t + 1) % len(pool.rand)] if t % 2 == 0 else pool.ones
        cv = pool.comp[v]
        left = full(cv)
        left[c] = pool.flip[cv]
        rows.append((left, full(v)))
    rows.append((rng.integers(0, P, cols), rng.integers(0, P, cols)))
    s = np.array(pool.single)
    rows.append((s[rng.integers(0, len(s), cols)], s[rng.integers(0, len(s), cols)]))
    rows.append((rng.integers(0, P, cols), rng.integers(0, P, cols)))
    return rows


# ------------------------------------------------------------------------------------------------ case table --
@dataclass
class Case:
    name: str  # the kernel lb.last_search_kernel() must name
    engine: str  # lb.set_search_engine
    k: int
    flags: int
    free_bits: int  # declared to the search (top_bit_free) and kept clear in the pool
    rows: int  # rows per search
    cols: int
    drange: Optional[Tuple[int, int]] = None


def _tiles256(cols: int) -> int:
    return (cols + 255) // 256


def rows_for_mma(variant: int, dirs: int, cols: int, sms: int) -> int:
    """launch_search_mma takes variant 2 iff K is 4 or 8 and dirs * rows * ceil(cols / 256) >= 2 * SMs."""
    need = 2 * sms
    per_row = dirs * _tiles256(cols)
    if variant == 2:
        return -(-need // per_row)
    return max(1, min(6, (need - 1) // per_row))


def case_table(sms: int):
    cases = []
    for k in KS:
        for flags in range(4):
            cases.append(Case(f"popc<K={k},flags={flags}>", "popc", k, flags, flags % 3, 6, 777))
    ranges = [(0, 63), (-40, 200), (5, 5), (-1499, 1000)]
    for k in KS:
        for flags in range(4):
            cases.append(Case(f"range<K={k},flags={flags}>", "auto", k, flags, 0, 6, 1500, ranges[(k + flags) % len(ranges)]))
    for cols in (COL_LIMIT_MMA, 1001):
        for k in (4, 8):
            for flags in range(4):
                dirs = 2 if flags & FLAG_CONSISTENCY else 1
                for ct in (0, 1):
                    for v in (1, 2):
                        rows = rows_for_mma(v, dirs, cols, sms)
                        name = f"mma{v}<K={k},nodupes={flags & 1},ct={ct},dirs={dirs}>"
                        cases.append(Case(name, "auto", k, flags, ct, rows, cols))
            cases.append(Case(f"mma3<K={k},nodupes=0,ct=2,onepass=1>", "auto", k, FLAG_CONSISTENCY, 2, 4, cols))
        for k in (12, 16):
            for flags in range(4):
                dirs = 2 if flags & FLAG_CONSISTENCY else 1
                cases.append(Case(f"mma1<K={k},nodupes={flags & 1},ct=0,dirs={dirs}>", "auto", k, flags, flags % 3, 3, cols))
    return cases


def expected_kernel_names():
    names = {f"popc<K={k},flags={f}>" for k in KS for f in range(4)}
    names |= {f"range<K={k},flags={f}>" for k in KS for f in range(4)}
    for v in (1, 2):
        names |= {f"mma{v}<K={k},nodupes={f & 1},ct={ct},dirs={2 if f & 2 else 1}>" for k in (4, 8) for f in range(4) for ct in (0, 1)}
    names |= {f"mma1<K={k},nodupes={f & 1},ct=0,dirs={2 if f & 2 else 1}>" for k in (12, 16) for f in range(4)}
    names |= {f"mma3<K={k},nodupes=0,ct=2,onepass=1>" for k in (4, 8)}
    return names


def _predicted_variant(case: Case, sms: int) -> Optional[int]:
    """The kernel family launch_search_mma picks for this case, restated (None: not the tensor-core engine)."""
    if case.engine != "auto" or case.drange is not None or case.k not in (4, 8, 12, 16):
        return None
    if case.k in (4, 8) and case.flags == FLAG_CONSISTENCY and case.free_bits >= 2:
        return 3
    dirs = 2 if case.flags & FLAG_CONSISTENCY else 1
    return 2 if case.k in (4, 8) and dirs * case.rows * _tiles256(case.cols) >= 2 * sms else 1


# ----------------------------------------------------------------------------------------------- CPU tests --
@pytest.mark.parametrize("k,free_bits", [(1, 0), (2, 1), (4, 2), (8, 0), (12, 1), (16, 2)])
@pytest.mark.parametrize("flags", range(4))
@pytest.mark.parametrize("drange", [None, (0, 9), (-6, 3), (4, 4), (50, 60), (-3, 20)])
def test_reference_keys_equal_brute_force(k, free_bits, flags, drange):
    rng = np.random.default_rng(100 * k + 10 * flags + free_bits)
    cols = 37  # (50, 60): every window empty
    pool = make_pool(k, free_bits, seed=k)
    prow = pattern_rows(pool, cols, rng)
    idx0 = np.stack([a for a, _ in prow])
    idx1 = np.stack([b for _, b in prow])
    want = brute_keys(pool.words[idx0], pool.words[idx1], flags, drange)
    got = reference_keys(idx0, idx1, pool.words, flags, drange)
    assert set(n for n, v in got.items() if v is not None) == set(n for n, v in want.items() if v is not None)
    assert_keys_equal(got, want, f"K={k} flags={flags} range={drange}")
    if drange == (50, 60):
        assert (got["fwd_first"] == KEY_NONE).all() and (got["fwd_last"] == KEY_NONE).all()


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("free_bits", [0, 1, 2])
def test_pools_reach_the_usable_cost_limits(k, free_bits):
    pool = make_pool(k, free_bits, seed=7)
    B = 32 * k - free_bits
    assert pool.bits == B
    assert popcount_words(pool.words[pool.ones]) == B
    if free_bits:
        assert not (pool.words[:, -1] >> np.uint32(32 - free_bits)).any()  # the declared free bits are clear
    for i, c in pool.comp.items():
        assert popcount_words(pool.words[i] ^ pool.words[c]) == B
    for i, f in pool.flip.items():
        assert popcount_words(pool.words[i] ^ pool.words[f]) == 1
    cols = 8192
    rows = pattern_rows(pool, cols, np.random.default_rng(k))
    keys = reference_keys(np.stack([a for a, _ in rows]), np.stack([b for _, b in rows]), pool.words, 3)
    cost = keys["fwd_first"] >> np.uint32(16)
    assert cost[0].min() == B and cost[2].max() == 0  # all ties at B, all ties at 0
    col = keys["fwd_first"][4] & np.uint32(0xFFFF)  # the first planted forward minimum, at column 0
    assert (cost[4] == B - 1).all() and (col == 0).all()


def test_case_table_reaches_every_kernel_name():
    want = expected_kernel_names()
    assert len(want) == 24 + 24 + 24 + 16 + 2
    for sms in (148, 132, 160, 96):
        cases = case_table(sms)
        names = {c.name for c in cases}
        assert names == want, sorted(names ^ want)
        for c in cases:
            fam = c.name.split("<")[0]
            v = _predicted_variant(c, sms)
            if fam.startswith("mma"):
                assert v == int(fam[3]), (sms, c)
                assert c.cols <= COL_LIMIT_MMA and c.rows >= 1
            else:
                assert v is None, c
    mma = [c for c in case_table(148) if c.name.startswith("mma")]
    assert {c.name for c in mma if c.cols == COL_LIMIT_MMA} == {n for n in want if n.startswith("mma")}


# ---------------------------------------------------------------------------------------- whole-match scenes --
def degenerate_scene(n: int, dtype, rows: int, cols: int, seed: int, disparity: int = 7):
    """Random texture with a constant disparity, overlaid with narrow bands of degenerate stacks. Left pixel x shows
    what right pixel x - disparity shows. Bands, varied per row: constant 0 / maximum / mid-grey on both sides, the left
    only or the right only; strictly monotone stacks; stacks alternating 0 and the maximum; stacks mid + 2t - (n - 1)
    (variance exactly n (n^2 - 1) / 3, exact in float); right an affine image (2 v + 3) or the complement (max - v) of
    the left; zero or saturated right neighbours of a match (the subpixel interpolation's wrap)."""
    rng = np.random.default_rng(seed)
    top = np.iinfo(dtype).max
    mid = top // 2
    d = disparity
    S = rng.integers(0, top + 1, size=(n, rows, cols + d), dtype=np.int64)
    t = np.arange(n)[:, None]
    kinds = ["c0", "cmax", "cmid", "mono", "alt", "exactvar", "l0", "rmax", "lmid", "affine", "anti", "nb0", "nbmax", "rand"]
    side = []  # side-only edits, applied after slicing: (kind, row, s0, w)
    x = 2
    band = 0
    while x + 4 < cols:
        w = 1 + band % 3
        for r in range(rows):
            kind = kinds[(band + r) % len(kinds)]
            sl = (slice(None), r, slice(x, x + w))
            if kind == "c0":
                S[sl] = 0
            elif kind == "cmax":
                S[sl] = top
            elif kind == "cmid":
                S[sl] = mid
            elif kind == "mono":
                S[sl] = (t * top) // (n - 1)
            elif kind == "alt":
                S[sl] = np.where(t % 2 == 0, 0, top)
            elif kind == "exactvar":
                S[sl] = mid + 2 * t - (n - 1)
            elif kind == "affine":
                S[sl] = rng.integers(0, (top - 3) // 2 + 1, size=(n, w))
                side.append((kind, r, x, w))
            else:
                side.append((kind, r, x, w))
        x += w + 3 + band % 4
        band += 1
    L = S[:, :, :cols].copy()
    R = S[:, :, d:].copy()
    for kind, r, s0, w in side:
        rs = slice(max(s0 - d, 0), max(s0 - d + w, 0))  # the right columns that show S columns s0 .. s0 + w - 1
        ss = slice(s0 + (rs.start - (s0 - d)), s0 + w)
        if kind == "l0":
            L[:, r, s0:s0 + w] = 0
        elif kind == "rmax":
            R[:, r, rs] = top
        elif kind == "lmid":
            L[:, r, s0:s0 + w] = mid
        elif kind == "affine":
            R[:, r, rs] = 2 * S[:, r, ss] + 3
        elif kind == "anti":
            R[:, r, rs] = top - S[:, r, ss]
        elif kind in ("nb0", "nbmax"):
            v = 0 if kind == "nb0" else top
            for c in (s0 - d - 1, s0 - d + w):
                if 0 <= c < cols:
                    R[:, r, c] = v
    assert L.min() >= 0 and L.max() <= top and R.min() >= 0 and R.max() <= top
    return L.astype(dtype), R.astype(dtype)


def exact_min_variance(n: int) -> float:
    """A float32 min_variance whose product with n, in float32 as the library and the oracle form it, is exactly the
    variance sum n (n^2 - 1) / 3 of the scene's exactvar stacks."""
    var = n * (n * n - 1) // 3
    m = np.float32(var / n)
    for c in (m, np.nextafter(m, np.float32(0)), np.nextafter(m, np.float32(np.inf))):
        if np.float32(c) * np.float32(n) == np.float32(var) and float(np.float32(var)) == var:
            return float(c)
    raise AssertionError(f"no float32 min_variance reaches {var} for n = {n}")


def exact_nxc(left, right, raw, min_variance=None):
    """The NXC of every pixel the integer-mode refine evaluates (raw disparity valid, partner inside the row), from the
    integer sums at 40 significant digits: num / sqrt(den0 den1) with num = n S01 - S0 S1, den = n Sxx - Sx^2.
    NaN for zero variance (0 / 0); with min_variance, -1 where a variance sum is below min_variance * n (float32).
    -> (nxc float64 [rows, cols] with NaN where not evaluated, evaluated mask, variance sums of both sides)."""
    n, rows, cols = left.shape
    c = np.arange(cols)[None, :]
    c1 = c - raw.astype(np.int64)
    ev = (raw != -32768) & (c1 >= 0) & (c1 < cols)
    r_idx = np.broadcast_to(np.arange(rows)[:, None], (rows, cols))
    a = left.astype(np.int64)
    b = right.astype(np.int64)[:, r_idx, np.clip(c1, 0, cols - 1)]
    s0, s1 = a.sum(0), b.sum(0)
    num = n * (a * b).sum(0) - s0 * s1
    den0 = n * (a * a).sum(0) - s0 * s0
    den1 = n * (b * b).sum(0) - s1 * s1
    mvn = None if min_variance is None else float(np.float32(min_variance) * np.float32(n))
    out = np.full((rows, cols), np.nan)
    with localcontext() as ctx:
        ctx.prec = 40
        for r, cc in zip(*np.nonzero(ev)):
            if mvn is not None and (Decimal(int(den0[r, cc])) < Decimal(mvn) * n or Decimal(int(den1[r, cc])) < Decimal(mvn) * n):
                out[r, cc] = -1.0
            elif den0[r, cc] == 0 or den1[r, cc] == 0:
                out[r, cc] = np.nan
            else:
                p = Decimal(int(den0[r, cc])) * Decimal(int(den1[r, cc]))
                out[r, cc] = float(Decimal(int(num[r, cc])) / p.sqrt())
    return out, ev, den0 / n, den1 / n


def check_against_exact_nxc(disp, corr, left, right, raw, kw, double, what):
    """Integer mode with a threshold: corrmap within 1e-12 (double) / 1e-5 (float) of the exact NXC, NaN for zero
    variance without min_variance (-1 with it), and the valid mask wherever the exact value is more than 1e-5 away from
    the threshold (a NaN correlation keeps the pixel valid: NaN < threshold is false)."""
    thr = kw["nxcorr_threshold"]
    mv = kw.get("min_variance")
    exact, ev, var0, var1 = exact_nxc(left, right, raw, mv)
    tol = 1e-12 if double else 1e-5
    if mv is not None:  # a variance sum next to min_variance * n may fall either way in float: skip those
        mvn = float(np.float32(mv) * np.float32(left.shape[0]))
        near = lambda v: (np.abs(v - mvn) <= 1e-3 * max(mvn, 1.0)) & (v != mvn)  # noqa: E731
        ev = ev & ~(near(var0) | near(var1))
    assert np.array_equal(np.isnan(corr[ev]), np.isnan(exact[ev])), f"{what}: NaN cells differ from the exact NXC"
    fin = ev & ~np.isnan(exact)
    err = np.abs(corr[fin].astype(np.float64) - exact[fin])
    assert err.max(initial=0) <= tol, f"{what}: corrmap off the exact NXC by {err.max():.3g}"
    if mv is None:
        zero_var = ev & ((var0 == 0) | (var1 == 0))
        assert np.isnan(corr[zero_var]).all()
    else:
        assert (corr[ev & ((var0 == 0) | (var1 == 0))] == -1).all()
    valid = ~np.isnan(disp) & (disp != -32768)
    decided = ev & (np.isnan(exact) | (np.abs(exact - thr) > 1e-5))
    want_valid = np.isnan(exact) | (exact >= thr)
    assert np.array_equal(valid[decided], want_valid[decided]), f"{what}: valid mask differs from the exact NXC"
    assert not valid[~ev].any(), f"{what}: a pixel without an evaluated correlation is valid"


NS = [2, 3, 4, 9, 17, 33, 65]
MATCH_CFGS = {
    "none": dict(nxcorr_threshold=None),
    "t0.5": dict(nxcorr_threshold=0.5),
    "t1": dict(nxcorr_threshold=1.0),
    # Consistency without no_dupes keeps first minima among ties: the only variant under which constant stacks match
    "t-1": dict(nxcorr_threshold=-1.0, consistency=True, max_lr_diff=1),
    "sub": dict(nxcorr_threshold=0.5, subpixel_step=0.25),
    "minvar": dict(nxcorr_threshold=0.5, min_variance="exact", consistency=True, max_lr_diff=2),
    "sub-minvar": dict(nxcorr_threshold=-1.0, subpixel_step=0.5, min_variance="exact", consistency=True, max_lr_diff=1),
    "cons": dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=1),
    "cons-nodupes": dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=1, no_dupes=True, subpixel_step=0.2),
}


def _resolve(kw, n):
    kw = dict(kw)
    if kw.get("min_variance") == "exact":
        kw["min_variance"] = exact_min_variance(n)
    return kw


def oracle_match(oracles, left, right, kw, double):
    """oracles.port.match, composed from its stages for a negative threshold (its match reads < 0 as no threshold)."""
    port = oracles.port
    thr = kw.get("nxcorr_threshold")
    if thr is None or thr >= 0:
        return port.match(left, right, double=double, **kw)
    rest = {k: v for k, v in kw.items() if k not in ("nxcorr_threshold", "subpixel_step", "min_variance")}
    raw, _ = port.match(left, right, nxcorr_threshold=None, **rest)
    disp, corr = port.agree(raw, left, right, thr, kw.get("subpixel_step"), kw.get("min_variance"), double=double)
    return (disp.astype(np.float32) if kw.get("subpixel_step") is None else disp), corr


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)


def _raw(oracles, left, right, kw):
    rest = {k: v for k, v in kw.items() if k not in ("nxcorr_threshold", "subpixel_step", "min_variance")}
    return oracles.port.match(left, right, nxcorr_threshold=None, **rest)[0]


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_oracle_correlation_is_the_exact_nxc(oracles, n, dtype):
    """The oracle's integer-mode refine on the degenerate scenes, float and double, against the exact NXC."""
    left, right = degenerate_scene(n, dtype, 16, 150, seed=n)
    for name in ("t0.5", "t1", "t-1", "minvar", "cons"):
        kw = _resolve(MATCH_CFGS[name], n)
        raw = _raw(oracles, left, right, kw)
        for double in (False, True):
            disp, corr = oracle_match(oracles, left, right, kw, double)
            check_against_exact_nxc(disp, corr, left, right, raw, kw, double, f"oracle {name} double={double}")


def test_scene_has_its_degenerate_stacks(oracles):
    n = 9
    left, right = degenerate_scene(n, np.uint8, 16, 150, seed=1)
    var_l = left.astype(np.int64).var(axis=0)
    var_r = right.astype(np.int64).var(axis=0)
    assert (var_l == 0).sum() > 50 and (var_r == 0).sum() > 50
    assert ((var_l == 0) & (var_r == 0)).any() and ((var_l == 0) & (var_r > 0)).any()
    kw = _resolve(MATCH_CFGS["minvar"], n)
    raw = _raw(oracles, left, right, kw)
    exact, ev, v0, v1 = exact_nxc(left, right, raw, kw["min_variance"])
    mvn = float(np.float32(kw["min_variance"]) * np.float32(n))
    assert (ev & ((v0 == mvn) | (v1 == mvn))).any(), "no evaluated pixel with a variance exactly at min_variance * n"
    exact, ev, _, _ = exact_nxc(left, right, raw)
    assert np.isnan(exact[ev]).any() and (exact[ev] == 1).any(), "no zero-variance or perfectly correlated match"


# ----------------------------------------------------------------------------------------------- GPU tests --
def _pitched(d):
    import torch

    rows, cols, k = d.shape
    buf = np.zeros((rows, (cols * k + 3) // 4 * 4), dtype=np.uint32)
    buf[:, : cols * k] = d.reshape(rows, cols * k)
    return torch.from_numpy(buf.view(np.int32)).cuda()


def _cuda(a):
    import torch

    if a.dtype == np.uint16:
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def sms(handle):
    import torch

    for var in ("BICOS_B200_MMA_VARIANT", "BICOS_B200_MMA_COLTERM"):
        if os.environ.get(var):
            pytest.skip(f"{var} overrides the kernel choice these tests assert")
    return torch.cuda.get_device_properties(0).multi_processor_count


def run_search(handle, pool: Pool, idx0, idx1, k, flags, free_bits, drange, engine="auto"):
    rows, cols = idx0.shape
    lb.set_search_engine(engine)
    try:
        keys = handle.search(_pitched(pool.words[idx0]), _pitched(pool.words[idx1]), k, cols, flags, top_bit_free=free_bits,
                             disparity_range=drange)
        kernel = lb.last_search_kernel()
    finally:
        lb.set_search_engine("auto")
    got = dict(zip(("fwd_first", "fwd_last", "rev_first", "rev_last"),
                   (t.cpu().numpy().view(np.uint32) if t is not None else None for t in keys)))
    return got, kernel


def check_case(handle, case: Case, seed: int):
    """All pattern rows of the case's pool, `case.rows` per search."""
    rng = np.random.default_rng(seed)
    pool = make_pool(case.k, case.free_bits, seed)
    prow = pattern_rows(pool, case.cols, rng)
    nb = -(-len(prow) // case.rows)
    while len(prow) < nb * case.rows:  # fill the last search with random rows
        P = len(pool.words)
        prow.append((rng.integers(0, P, case.cols), rng.integers(0, P, case.cols)))
    for b in range(nb):
        part = prow[b * case.rows:(b + 1) * case.rows]
        idx0, idx1 = np.stack([a for a, _ in part]), np.stack([c for _, c in part])
        got, kernel = run_search(handle, pool, idx0, idx1, case.k, case.flags, case.free_bits, case.drange, case.engine)
        assert kernel == case.name, f"dispatched {kernel}, expected {case.name}"
        want = reference_keys(idx0, idx1, pool.words, case.flags, case.drange)
        assert_keys_equal(got, want, f"{case.name} cols={case.cols} rows {b * case.rows}..")


def _case_ids():
    return [f"{c.name}-{c.cols}" for c in case_table(148)]


@pytest.mark.gpu
@pytest.mark.parametrize("index", range(len(case_table(148))), ids=_case_ids())
def test_search_kernel_extremes(handle, sms, index):
    case = case_table(sms)[index]
    check_case(handle, case, seed=1000 + index)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [4, 8])
@pytest.mark.parametrize("flags", range(4))
def test_auto_engine_takes_popc_past_8192_columns(handle, k, flags):
    cols = COL_LIMIT_MMA + 1
    rng = np.random.default_rng(k + flags)
    pool = make_pool(k, 2, seed=k)
    prow = pattern_rows(pool, cols, rng)[:3] + pattern_rows(pool, cols, rng)[-3:]
    idx0, idx1 = np.stack([a for a, _ in prow]), np.stack([b for _, b in prow])
    got, kernel = run_search(handle, pool, idx0, idx1, k, flags, 2, None)
    assert kernel == f"popc<K={k},flags={flags}>"
    assert_keys_equal(got, reference_keys(idx0, idx1, pool.words, flags), f"auto at {cols} columns")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 16])
def test_popc_at_32767_columns(handle, k):
    cols = COL_LIMIT
    rng = np.random.default_rng(k)
    pool = make_pool(k, 0, seed=k)
    # all ties at B, a unique forward and a unique reverse minimum in the last column
    prow = pattern_rows(pool, cols, rng)
    last = len(min_columns(cols)) - 1
    picks = [0, 4 + 2 * last, 5 + 2 * last]
    for r0 in (0, 1):
        part = [prow[picks[0]], prow[picks[1 + r0]]]
        idx0, idx1 = np.stack([a for a, _ in part]), np.stack([b for _, b in part])
        got, kernel = run_search(handle, pool, idx0, idx1, k, 3, 0, None, engine="popc")
        assert kernel == f"popc<K={k},flags=3>"
        assert_keys_equal(got, reference_keys(idx0, idx1, pool.words, 3), f"popc K={k} at {cols} columns")


@pytest.mark.gpu
@pytest.mark.parametrize("k,drange", [(1, (-10, 50)), (16, (-10, 50)), (16, (-30000, 30000)), (4, (-30000, 30000)),
                                      (8, (100, 32766))])
@pytest.mark.parametrize("flags", [FLAG_NODUPES | FLAG_CONSISTENCY, 0])
def test_range_at_32767_columns(handle, k, drange, flags):
    """A narrow window, and wide windows that do not cover the row: the kernel stages the right row in chunks."""
    cols = COL_LIMIT
    rng = np.random.default_rng([k, abs(drange[0]), flags])
    pool = make_pool(k, 0, seed=k)
    prow = pattern_rows(pool, cols, rng)
    nmin = len(min_columns(cols))
    part = [prow[0], prow[4 + 2 * (nmin - 1)], prow[5 + 2 * (nmin - 2)], prow[-3]]
    idx0, idx1 = np.stack([a for a, _ in part]), np.stack([b for _, b in part])
    got, kernel = run_search(handle, pool, idx0, idx1, k, flags, 0, drange)
    assert kernel == f"range<K={k},flags={flags}>"
    assert_keys_equal(got, reference_keys(idx0, idx1, pool.words, flags, drange), f"range {drange} K={k}")


def _check_match(handle, oracles, left, right, kw, double, what):
    disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=double, **kw))
    got_d = disp.cpu().numpy()
    want_d, want_c = oracle_match(oracles, left, right, kw, double)
    assert got_d.dtype == want_d.dtype, what
    if kw.get("nxcorr_threshold") is None:
        assert corr is None and np.array_equal(got_d, want_d), f"{what}: {(got_d != want_d).sum()} disparities differ"
        return got_d, None
    got_c = corr.cpu().numpy()
    if not double:
        assert _same(got_d, want_d), f"{what}: disparity differs from the oracle at {np.argwhere(got_d != want_d)[:3].tolist()}"
        assert _same(got_c, want_c), f"{what}: corrmap differs from the oracle"
        return got_d, got_c
    thr = kw["nxcorr_threshold"]
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c)), f"{what}: NaN cells of the corrmap differ"
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= 1e-12, f"{what}: double corrmap"
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    edge = np.abs(np.nan_to_num(want_c, nan=9.0) - thr) < 1e-6
    assert np.array_equal(invalid_g | edge, invalid_w | edge), f"{what}: valid masks differ"
    both = ~(invalid_w | invalid_g)
    assert np.array_equal(got_d[both], want_d[both]) if kw.get("subpixel_step") is None else \
        np.max(np.abs(got_d[both] - want_d[both]), initial=0) <= 1e-3
    return got_d, got_c


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
@pytest.mark.parametrize("cfg", list(MATCH_CFGS))
def test_match_on_degenerate_stacks(handle, oracles, n, dtype, cfg):
    """The whole match against the oracle (float bit for bit, double within 1e-12), and in integer mode with a
    threshold against the exact NXC."""
    left, right = degenerate_scene(n, dtype, 16, 150, seed=n + (0 if dtype == np.uint8 else 100))
    kw = _resolve(MATCH_CFGS[cfg], n)
    raw = None
    for double in ((False,) if kw["nxcorr_threshold"] is None else (False, True)):
        got_d, got_c = _check_match(handle, oracles, left, right, kw, double, f"n={n} {np.dtype(dtype).name} {cfg} double={double}")
        if got_c is not None and kw.get("subpixel_step") is None:
            raw = _raw(oracles, left, right, kw) if raw is None else raw
            check_against_exact_nxc(got_d, got_c, left, right, raw, kw, double, f"kernel {cfg} n={n} double={double}")
        elif got_c is not None and kw.get("min_variance") is not None:
            # subpixel with min_variance: a zero-variance pixel keeps the initial best of -1
            raw = _raw(oracles, left, right, kw) if raw is None else raw
            _, ev, v0, v1 = exact_nxc(left, right, raw)
            c = np.arange(left.shape[2])[None, :] - raw
            inner = ev & (c > 0) & (c < left.shape[2] - 1)
            zero = inner & (v0 == 0)
            assert zero.any() and (got_c[zero] == -1).all()


@pytest.mark.gpu
def test_match_past_8192_columns(handle, oracles):
    left, right = degenerate_scene(33, np.uint8, 3, COL_LIMIT_MMA + 1, seed=8193)
    kw = dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=1)
    _check_match(handle, oracles, left, right, kw, False, "8193 columns")
    assert lb.last_search_kernel() == "popc<K=4,flags=2>"  # 4 n - 6 = 126 descriptor bits
