"""Per-pixel disparity windows: bicos_b200_search_windows, bicos_b200_match_windows and bicos_b200_windows_from_disparity.

window_keys() restates the key arrays of include/bicos_b200.h for window maps: every in-window pair (left i, right j)
with min[r, i] <= i - j <= max[r, i], clipped to the row, as an explicit list; the forward keys are per-pixel minima over
each pixel's contiguous run of pairs, the reverse keys a scatter-min (np.minimum.at) over the same pairs, because the
left columns that reach one right column need not be contiguous. postfilter() turns keys into the raw disparity the
refine starts from. CPU: the restatement against a brute force over the full cost matrix, against reference_keys() of
test_search_extremes.py for constant maps, and against _bicos_range() of test_disparity_range.py; the prior-to-windows
rule against hand-computed values. GPU: the stage bit for bit against the restatement, the equivalences with the range
and the full row, whole matches against the oracle's refinement, and every entry point (C ABI, C++, CLI).
"""

import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config, synth

from test_disparity_range import _bicos_range, _read_output, _write_input
from test_search_extremes import reference_keys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAG_NODUPES, FLAG_CONSISTENCY = 1, 2
KEY_NONE = 0xFFFFFFFF
INVALID = -32768
NAMES = ("fwd_first", "fwd_last", "rev_first", "rev_last")


# ------------------------------------------------------------------------------------------ restatement --
def pool_cost(idx0, idx1, pool):
    """cost(r, i, j) for descriptors pool[idx0] (left) and pool[idx1] (right), idx [rows, cols] into pool [P, K]."""
    table = np.bitwise_count(pool[:, None, :] ^ pool[None, :, :]).sum(axis=-1, dtype=np.int64)
    return lambda r, i, j: table[idx0[r, i], idx1[r, j]]


def desc_cost(d0, d1):
    """cost(r, i, j) for [rows, cols, K] uint32 descriptors."""
    return lambda r, i, j: np.bitwise_count(d0[r, i] ^ d1[r, j]).sum(axis=-1, dtype=np.int64)


def window_pairs(wmin_row, wmax_row, cols):
    """The in-window pairs of one row, grouped by left pixel: (i, j) arrays and each pixel's [lo, hi] (empty if lo > hi)."""
    x = np.arange(cols, dtype=np.int64)
    lo = np.maximum(x - wmax_row.astype(np.int64), 0)
    hi = np.minimum(x - wmin_row.astype(np.int64), cols - 1)
    n = np.maximum(hi - lo + 1, 0)
    i = np.repeat(x, n)
    start = np.repeat(np.cumsum(n) - n, n)
    j = np.repeat(lo, n) + np.arange(int(n.sum()), dtype=np.int64) - start
    return i, j, n


def window_keys(cost, rows, cols, wmin, wmax, flags):
    """The key arrays bicos_b200_search_windows fills (fwd_last always; rev_* with CONSISTENCY, rev_last with both)."""
    nodupes, cons = bool(flags & FLAG_NODUPES), bool(flags & FLAG_CONSISTENCY)
    out = {"fwd_first": np.full((rows, cols), KEY_NONE, np.uint64), "fwd_last": np.full((rows, cols), KEY_NONE, np.uint64),
           "rev_first": np.full((rows, cols), KEY_NONE, np.uint64) if cons else None,
           "rev_last": np.full((rows, cols), KEY_NONE, np.uint64) if nodupes and cons else None}
    for r in range(rows):
        i, j, n = window_pairs(wmin[r], wmax[r], cols)
        if len(i) == 0:
            continue
        c = cost(r, i, j).astype(np.uint64) << np.uint64(16)
        has = n > 0
        starts = (np.cumsum(n) - n)[has]
        ff = np.minimum.reduceat(c | j.astype(np.uint64), starts)
        out["fwd_first"][r, has] = ff
        if nodupes:
            out["fwd_last"][r, has] = np.minimum.reduceat(c | (65535 - j).astype(np.uint64), starts)
        else:
            out["fwd_last"][r, has] = (ff & np.uint64(0xFFFF0000)) | (np.uint64(65535) - (ff & np.uint64(0xFFFF)))
        if cons:
            np.minimum.at(out["rev_first"][r], j, c | i.astype(np.uint64))
            if nodupes:
                np.minimum.at(out["rev_last"][r], j, c | (65535 - i).astype(np.uint64))
    return {k: (v.astype(np.uint32) if v is not None else None) for k, v in out.items()}


def postfilter(keys, flags, max_lr):
    """The raw int16 disparity of bicos() on window keys: the first strict forward minimum (with NODUPES unique), with
    CONSISTENCY checked against the reverse minimum of the matched column (unique with NODUPES as well)."""
    ff, fl = keys["fwd_first"].astype(np.int64), keys["fwd_last"].astype(np.int64)
    rows, cols = ff.shape
    x = np.arange(cols)[None, :]
    best = ff & 0xFFFF
    ok = (ff != KEY_NONE) & ((65535 - (fl & 0xFFFF)) == best)
    out = np.full((rows, cols), INVALID, np.int16)
    if not flags & FLAG_CONSISTENCY:
        out[ok] = (x - best)[ok]
        return out
    b = np.where(ok, best, 0)
    rk = np.take_along_axis(keys["rev_first"].astype(np.int64), b, axis=1)
    rev = rk & 0xFFFF
    ok &= rk != KEY_NONE
    if flags & FLAG_NODUPES:
        rl = np.take_along_axis(keys["rev_last"].astype(np.int64), b, axis=1)
        ok &= (65535 - (rl & 0xFFFF)) == rev
    ok &= np.abs(x - rev) <= max_lr
    out[ok] = ((x + rev) // 2 - best)[ok]
    return out


def windows_restated(prior, margin, fallback=None):
    """bicos_b200_windows_from_disparity: (min, max) int16 maps from an int16 / float32 prior."""
    p = prior.astype(np.float64)
    if prior.dtype == np.int16:
        valid = prior != INVALID
    else:
        valid = np.isfinite(prior) & (prior != np.float32(-32768.0))
    fb = (-32768, 32767) if fallback is None else fallback
    with np.errstate(invalid="ignore"):
        lo = np.clip(np.floor(np.where(valid, p, 0.0)) - margin, -32768, 32767)
        hi = np.clip(np.ceil(np.where(valid, p, 0.0)) + margin, -32768, 32767)
    return np.where(valid, lo, fb[0]).astype(np.int16), np.where(valid, hi, fb[1]).astype(np.int16)


# --------------------------------------------------------------------------------------------- map kinds --
def make_windows(kind, rows, cols, rng):
    """int16 (min, max) maps of one kind."""
    shape = (rows, cols)
    x = np.arange(cols)[None, :]
    r = np.arange(rows)[:, None]
    if kind == "constant":
        lo, hi = sorted(int(v) for v in rng.integers(-40, 90, 2))
        return np.full(shape, lo, np.int16), np.full(shape, hi, np.int16)
    if kind == "tilted":  # a plane: bounds move with the row and the column
        c = 10 + 0.02 * x + 3 * r
        return (np.floor(c) - 4).astype(np.int16) + np.zeros(shape, np.int16), (np.ceil(c) + 6).astype(np.int16) + np.zeros(shape, np.int16)
    if kind == "random":
        lo = rng.integers(-60, 80, shape)
        return lo.astype(np.int16), (lo + rng.integers(0, 40, shape)).astype(np.int16)
    if kind == "partly_empty":  # random windows, a third of them empty (min > max)
        lo = rng.integers(-20, 60, shape)
        hi = lo + rng.integers(0, 30, shape)
        empty = rng.random(shape) < 1 / 3
        return lo.astype(np.int16), np.where(empty, lo - 1 - rng.integers(0, 5, shape), hi).astype(np.int16)
    if kind == "full_row_lane":  # narrow windows, one lane per warp (per CTA past 9000 columns) covering the row: chunks
        lo = rng.integers(0, 8, shape)
        wmin, wmax = lo.astype(np.int16), (lo + 3).astype(np.int16)
        lane = (x % (32 if cols <= 9000 else 128) == 5) & np.ones(shape, bool)
        return np.where(lane, -32768, wmin).astype(np.int16), np.where(lane, 32767, wmax).astype(np.int16)
    if kind == "disjoint":  # neighbouring lanes far apart: the warp's intersection is empty
        far = np.where(x % 2 == 0, -300, 300) + np.zeros(shape, np.int64)
        return (far - 2).astype(np.int16), (far + 2).astype(np.int16)
    if kind == "extreme":  # bounds at the int16 limits and beyond +-cols: empty, narrow and (a few) covering windows
        pick = rng.integers(0, 5, shape)
        lo = np.choose(pick, [32767, cols + 3, 0, -cols - 7, 3])
        hi = np.choose(pick, [32767, cols + 3, 5, -cols - 7, -32768])
        wide = rng.random(shape) < min(0.3, 40 / cols)
        lo = np.where(wide, np.choose(rng.integers(0, 2, shape), [-32768, -cols - 7]), lo)
        hi = np.where(wide, np.choose(rng.integers(0, 2, shape), [32767, cols + 3]), hi)
        return np.clip(lo, -32768, 32767).astype(np.int16), np.clip(hi, -32768, 32767).astype(np.int16)
    raise ValueError(kind)


MAP_KINDS = ("constant", "tilted", "random", "partly_empty", "full_row_lane", "disjoint", "extreme")


# ------------------------------------------------------------------------------------------------- CPU --
@pytest.mark.parametrize("k", [1, 2, 4])
@pytest.mark.parametrize("flags", range(4))
def test_window_keys_equal_brute_force(k, flags):
    rng = np.random.default_rng(10 * k + flags)
    rows, cols = 3, 45
    d0 = rng.integers(0, 4, size=(rows, cols, k)).astype(np.uint32)
    d1 = rng.integers(0, 4, size=(rows, cols, k)).astype(np.uint32)
    d0[:, 10:30] = d1[:, 4:24]
    for kind in MAP_KINDS:
        wmin, wmax = make_windows(kind, rows, cols, rng)
        got = window_keys(desc_cost(d0, d1), rows, cols, wmin, wmax, flags)
        want = {name: np.full((rows, cols), KEY_NONE, np.uint32) for name in NAMES}
        for r in range(rows):
            cost = np.bitwise_count(d0[r][:, None, :] ^ d1[r][None, :, :]).sum(axis=-1, dtype=np.int64)  # [left, right]
            dd = np.arange(cols)[:, None] - np.arange(cols)[None, :]
            inw = (dd >= wmin[r][:, None].astype(np.int64)) & (dd <= wmax[r][:, None].astype(np.int64))
            for c in range(cols):
                if inw[c].any():
                    m = np.where(inw[c], cost[c], 1 << 40)
                    at = np.flatnonzero(m == m.min())
                    want["fwd_first"][r, c] = int(m.min()) << 16 | int(at[0])
                    want["fwd_last"][r, c] = int(m.min()) << 16 | (65535 - int(at[-1] if flags & FLAG_NODUPES else at[0]))
                if inw[:, c].any():
                    m = np.where(inw[:, c], cost[:, c], 1 << 40)
                    at = np.flatnonzero(m == m.min())
                    want["rev_first"][r, c] = int(m.min()) << 16 | int(at[0])
                    want["rev_last"][r, c] = int(m.min()) << 16 | (65535 - int(at[-1]))
        for name in NAMES:
            if got[name] is None:
                assert name.startswith("rev") and (not flags & FLAG_CONSISTENCY or (name == "rev_last" and flags != 3))
                continue
            assert np.array_equal(got[name], want[name]), (kind, name)


@pytest.mark.parametrize("k", [1, 2, 4])
@pytest.mark.parametrize("flags", range(4))
def test_constant_windows_are_the_range(k, flags):
    rng = np.random.default_rng(k * 7 + flags)
    pool = rng.integers(0, 1 << 5, size=(9, k)).astype(np.uint32)
    rows, cols = 3, 300
    idx0, idx1 = rng.integers(0, len(pool), (rows, cols)), rng.integers(0, len(pool), (rows, cols))
    for drange in ((0, 9), (-6, 3), (4, 4), (50, 60), (-3, 20), (-32768, 32767), (310, 400)):
        wmin, wmax = (np.full((rows, cols), v, np.int16) for v in drange)
        got = window_keys(pool_cost(idx0, idx1, pool), rows, cols, wmin, wmax, flags)
        want = reference_keys(idx0, idx1, pool, flags, drange)
        for name in NAMES:
            if want[name] is not None:
                assert np.array_equal(got[name], want[name]), (drange, name)
        if drange == (-32768, 32767):  # covering maps: the unranged keys
            full = reference_keys(idx0, idx1, pool, flags)
            for name in ("fwd_first", "rev_first", "rev_last") + (("fwd_last",) if flags & FLAG_NODUPES else ()):
                if full[name] is not None:
                    assert np.array_equal(got[name], full[name]), name


@pytest.mark.parametrize("flags", [FLAG_NODUPES, FLAG_CONSISTENCY, FLAG_NODUPES | FLAG_CONSISTENCY])
def test_postfilter_of_constant_windows_is_the_ranged_bicos(flags):
    rng = np.random.default_rng(flags)
    rows, cols, k = 3, 60, 2
    d0 = rng.integers(0, 8, size=(rows, cols, k)).astype(np.uint32)
    d1 = rng.integers(0, 8, size=(rows, cols, k)).astype(np.uint32)
    d0[:, 10:40] = d1[:, 3:33]
    for lo, hi in ((0, 10), (-5, 5), (3, 3), (-20, -3), (60, 70), (-1000, 1000)):
        wmin, wmax = np.full((rows, cols), lo, np.int16), np.full((rows, cols), hi, np.int16)
        got = postfilter(window_keys(desc_cost(d0, d1), rows, cols, wmin, wmax, flags), flags, 2)
        assert np.array_equal(got, _bicos_range(d0, d1, flags, 2, lo, hi)), (lo, hi)


def test_windows_restatement_by_hand():
    f = np.array([[3.0, 3.25, -2.5, np.nan, -32768.0, np.inf, -np.inf, 1e30, -1e30, 32767.5, -32767.5, 0.0]], np.float32)
    for margin in (0, 2, 32767):
        for fallback in (None, (5, 4), (-3, 9)):
            lo, hi = windows_restated(f, margin, fallback)
            fb = (-32768, 32767) if fallback is None else fallback
            for c, v in enumerate(f[0].tolist()):
                if math.isnan(v) or math.isinf(v) or v == -32768.0:
                    assert (lo[0, c], hi[0, c]) == fb, (v, margin, fallback)
                else:
                    assert lo[0, c] == max(-32768, min(32767, math.floor(v) - margin)), (v, margin)
                    assert hi[0, c] == max(-32768, min(32767, math.ceil(v) + margin)), (v, margin)
    i16 = np.array([[-32768, -32767, 0, 17, 32767]], np.int16)
    lo, hi = windows_restated(i16, 4, (1, 0))
    assert lo.tolist() == [[1, -32768, -4, 13, 32763]] and hi.tolist() == [[0, -32763, 4, 21, 32767]]


def test_config_struct_of_windows():
    from libbicos_b200.capi import CDisparityWindows

    assert ctypes.sizeof(CDisparityWindows) == 24
    assert "bicos_b200_match_windows" in lb.capi.EXPORTS


def test_windows_check_binary_is_built():
    assert os.path.exists(os.path.join(ROOT, "tests", "cpp", "build", "windows_check"))


# ------------------------------------------------------------------------------------------------- GPU --
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


def _maps(wmin, wmax, pad=0):
    """(min, max) int16 CUDA tensors, with `pad` extra elements per row (a padded pitch)."""
    import torch

    rows, cols = wmin.shape
    out = []
    for m in (wmin, wmax):
        t = torch.full((rows, cols + pad), 0x1234, dtype=torch.int16, device="cuda")
        t[:, :cols] = torch.from_numpy(np.ascontiguousarray(m)).cuda()
        out.append(t[:, :cols])
    return tuple(out)


def _keys_np(keys):
    return dict(zip(NAMES, (t.cpu().numpy().view(np.uint32) if t is not None else None for t in keys)))


def _assert_keys(got, want, what):
    for name in NAMES:
        if want[name] is None:
            continue
        g = got[name]
        assert g is not None, f"{what}: {name} missing"
        if not np.array_equal(g, want[name]):
            r, c = (int(v) for v in np.argwhere(g != want[name])[0])
            raise AssertionError(f"{what}: {name} differs at {(g != want[name]).sum()} pixels, first ({r}, {c}): "
                                 f"got {int(g[r, c]):#x}, want {int(want[name][r, c]):#x}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 4, 8, 12, 16])
@pytest.mark.parametrize("flags", range(4))
@pytest.mark.parametrize("cols", [97, 700, 1300, 9000, 32767])
def test_search_windows_stage_bit_exact(handle, k, flags, cols):
    rng = np.random.default_rng([k, flags, cols])
    pool = rng.integers(0, 1 << 4, size=(11, k)).astype(np.uint32)
    rows = 2 if cols > 9000 else 3
    idx0, idx1 = rng.integers(0, len(pool), (rows, cols)), rng.integers(0, len(pool), (rows, cols))
    d0, d1 = _pitched(pool[idx0]), _pitched(pool[idx1])
    cost = pool_cost(idx0, idx1, pool)
    for n, kind in enumerate(MAP_KINDS):
        wmin, wmax = make_windows(kind, rows, cols, rng)
        got = _keys_np(handle.search(d0, d1, k, cols, flags, windows=_maps(wmin, wmax, pad=3 * (n % 2))))
        assert lb.last_search_kernel() == f"windows<K={k},flags={flags}>"
        _assert_keys(got, window_keys(cost, rows, cols, wmin, wmax, flags), f"{kind} K={k} flags={flags} cols={cols}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,kw", [
    (33, np.uint8, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (33, np.uint8, dict(nxcorr_threshold=None)),
    (16, np.uint16, dict(nxcorr_threshold=0.9, mode_full=True, consistency=True, no_dupes=True)),
    (9, np.uint8, dict(nxcorr_threshold=0.8, subpixel_step=0.3, double=True)),
])
def test_constant_and_covering_windows_equal_range_and_full_row(handle, n, dtype, kw):
    import torch

    rows, cols = 48, 320
    left, right, _ = synth.make_stacks(n, 512, cols, dtype, seed=n + cols, row0=128, rows=rows)
    l, r = _cuda(left), _cuda(right)

    def same(a, b):
        if a is None or b is None:
            return a is None and b is None
        return torch.equal(a, b) if not a.dtype.is_floating_point else bool(((a == b) | (a.isnan() & b.isnan())).all())

    for drange in ((14, 77), (-8, 40)):
        want = handle.match(l, r, Config(disparity_range=drange, **kw))
        wmin, wmax = (torch.full((rows, cols), v, dtype=torch.int16, device="cuda") for v in drange)
        got = handle.match_windows(l, r, (wmin, wmax), Config(**kw))
        assert lb.last_search_kernel().startswith("windows<")
        assert same(got[0], want[0]) and same(got[1], want[1]), drange
    want = handle.match(l, r, Config(**kw))
    for lo, hi in ((-32768, 32767), (-cols, cols), (-(cols - 1), cols - 1)):
        wmin, wmax = (torch.full((rows, cols), v, dtype=torch.int16, device="cuda") for v in (lo, hi))
        got = handle.match_windows(l, r, (wmin, wmax), Config(**kw))
        assert same(got[0], want[0]) and same(got[1], want[1]), (lo, hi)
    wmin, wmax = (torch.full((rows, cols), v, dtype=torch.int16, device="cuda") for v in (5, 4))
    disp, corr = handle.match_windows(l, r, (wmin, wmax), Config(**kw))
    d = disp.cpu().numpy()
    assert bool(((d == INVALID) | np.isnan(d.astype(np.float64))).all())
    assert corr is None or bool(corr.isnan().all())


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 4, 16])
@pytest.mark.parametrize("flags", range(4))
def test_constant_window_keys_equal_range_keys(handle, k, flags):
    rng = np.random.default_rng(k + 10 * flags)
    rows, cols = 3, 1300
    d0 = _pitched(rng.integers(0, 8, size=(rows, cols, k)).astype(np.uint32))
    d1 = _pitched(rng.integers(0, 8, size=(rows, cols, k)).astype(np.uint32))
    for drange in ((14, 77), (-300, 900), (2000, 2100)):
        want = _keys_np(handle.search(d0, d1, k, cols, flags, disparity_range=drange))
        got = _keys_np(handle.search(d0, d1, k, cols, flags,
                                     windows=_maps(*(np.full((rows, cols), v, np.int16) for v in drange))))
        _assert_keys(got, want, f"constant {drange}")


def _oracle_windowed(oracles, left, right, wmin, wmax, kw, double):
    port = oracles.port
    full = kw.get("mode_full", False)
    d0, d1 = port.descriptors(left, full), port.descriptors(right, full)
    flags = (FLAG_CONSISTENCY | (FLAG_NODUPES if kw.get("no_dupes") else 0)) if kw.get("consistency") else FLAG_NODUPES
    rows, cols = wmin.shape
    raw = postfilter(window_keys(desc_cost(d0, d1), rows, cols, wmin, wmax, flags), flags, kw.get("max_lr_diff", 1))
    if kw.get("nxcorr_threshold") is None:
        return raw, None
    disp, corr = port.agree(raw, left, right, kw["nxcorr_threshold"], kw.get("subpixel_step"), kw.get("min_variance"), double=double)
    return (disp.astype(np.float32) if kw.get("subpixel_step") is None else disp), corr


MATCH_CASES = [
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0)),
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=None)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2, no_dupes=True)),
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, subpixel_step=0.1, consistency=True)),
    (9, np.uint8, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.3)),
    (17, np.uint16, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.15, min_variance=4.0)),
    (12, np.uint8, 32, 200, dict(nxcorr_threshold=0.7, mode_full=True, consistency=True, max_lr_diff=0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,rows,cols,kw", MATCH_CASES)
@pytest.mark.parametrize("maps", ["prior", "random", "partly_empty"])
@pytest.mark.parametrize("double", [False, True])
def test_windowed_match_parity(handle, oracles, n, dtype, rows, cols, kw, maps, double):
    if double and kw["nxcorr_threshold"] is None:
        pytest.skip("no correlation stage, no precision")
    rng = np.random.default_rng([n, cols, len(maps)])
    left, right, truth = synth.make_stacks(n, 512, cols, dtype, seed=11 * n + cols, row0=128, rows=rows)
    if maps == "prior":  # the true disparity +- 2, and no window in a band of columns (a region of interest)
        wmin, wmax = windows_restated(truth.astype(np.float32), 2)
        wmax[:, cols // 3: cols // 3 + 20] = wmin[:, cols // 3: cols // 3 + 20] - 1
    else:
        wmin, wmax = make_windows(maps, rows, cols, rng)
    want_d, want_c = _oracle_windowed(oracles, left, right, wmin, wmax, kw, double)
    disp, corr = handle.match_windows(_cuda(left), _cuda(right), _maps(wmin, wmax), Config(double=double, **kw))
    got_d = disp.cpu().numpy()
    assert got_d.dtype == want_d.dtype
    if want_d.dtype == np.int16:
        assert np.array_equal(got_d, want_d) and corr is None
        return
    got_c = corr.cpu().numpy()
    if not double:
        assert np.array_equal(got_d, want_d, equal_nan=True) and np.array_equal(got_c, want_c, equal_nan=True)
        return
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    edge = np.abs(np.nan_to_num(want_c, nan=9.0) - kw["nxcorr_threshold"]) < 1e-6
    assert np.array_equal(invalid_g | edge, invalid_w | edge), "valid masks differ"
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c))
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= 1e-12
    both = ~(invalid_w | invalid_g)
    assert np.max(np.abs(got_d[both] - want_d[both]), initial=0) <= 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
@pytest.mark.parametrize("shape,pad", [((1, 1), 0), ((7, 300), 5), ((64, 2048), 0), ((3, 32767), 1)])
def test_windows_from_disparity_exact(handle, dtype, shape, pad):
    import torch

    rng = np.random.default_rng(shape[1])
    rows, cols = shape
    if dtype == np.int16:
        prior = rng.integers(-32768, 32768, shape).astype(np.int16)
        prior[rng.random(shape) < 0.2] = INVALID
    else:
        prior = (rng.standard_normal(shape) * 80).astype(np.float32)
        special = np.array([np.nan, np.inf, -np.inf, -32768.0, 1e30, -1e30, 32767.5, 0.5], np.float32)
        mask = rng.random(shape) < 0.3
        prior[mask] = rng.choice(special, int(mask.sum()))
    src = torch.zeros((rows, cols + pad), dtype=torch.int16 if dtype == np.int16 else torch.float32, device="cuda")
    src[:, :cols] = torch.from_numpy(prior).cuda()
    for margin in (0, 3, 32767):
        for fallback in (None, (5, 4), (-7, 60)):
            out = _maps(np.zeros(shape, np.int16), np.zeros(shape, np.int16), pad=2)
            before = handle.kernel_launches
            lo, hi = handle.windows_from_disparity(src[:, :cols], margin, fallback, out=out)
            assert handle.kernel_launches == before + 1
            want = windows_restated(prior, margin, fallback)
            assert np.array_equal(lo.cpu().numpy(), want[0]) and np.array_equal(hi.cpu().numpy(), want[1]), (margin, fallback)


@pytest.mark.gpu
def test_windows_errors_launch_nothing(handle):
    import torch

    rows, cols = 16, 64
    left, right, _ = synth.make_stacks(9, 32, cols, np.uint8, seed=3, rows=rows)
    l, r = _cuda(left), _cuda(right)
    wmin = torch.zeros((rows, cols), dtype=torch.int16, device="cuda")
    wmax = torch.full((rows, cols), 20, dtype=torch.int16, device="cuda")
    L = lb.lib()
    ccfg = Config().to_c()
    p0, n, _, _, pitch, depth = handle._stack_info(l)
    p1 = handle._stack_info(r)[0]
    disp = torch.empty((rows, cols), dtype=torch.float32, device="cuda")
    st = handle._stream()

    def call(win, cfg=ccfg):
        return L.bicos_b200_match_windows(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(cfg),
                                          ctypes.byref(win) if win is not None else None, disp.data_ptr(), cols * 4, None, 0, st)

    from libbicos_b200.capi import CDisparityWindows

    before = handle.kernel_launches
    good = CDisparityWindows(wmin.data_ptr(), wmax.data_ptr(), cols * 2)
    for win, what in ((None, "null"), (CDisparityWindows(None, wmax.data_ptr(), cols * 2), "null"),
                      (CDisparityWindows(wmin.data_ptr(), None, cols * 2), "null"),
                      (CDisparityWindows(wmin.data_ptr(), wmax.data_ptr(), cols * 2 + 1), "pitch"),
                      (CDisparityWindows(wmin.data_ptr(), wmax.data_ptr(), cols * 2 - 2), "pitch")):
        assert call(win) == -1, what
        assert what in lb.lib().bicos_b200_last_error().decode()
    assert call(good, Config(disparity_range=(0, 9)).to_c()) == -1
    assert "exclude" in L.bicos_b200_last_error().decode()
    d = torch.zeros((rows, cols * 4), dtype=torch.int32, device="cuda")
    with pytest.raises(lb.BicosError, match="exclude"):
        handle.search(d, d, 4, cols, FLAG_NODUPES, disparity_range=(0, 1), windows=(wmin, wmax))
    keys = torch.empty((2, rows, cols), dtype=torch.int32, device="cuda")
    assert L.bicos_b200_search_windows(handle._h, d.data_ptr(), d.data_ptr(), 4, rows, cols, cols * 4, FLAG_NODUPES, keys[0].data_ptr(),
                                       keys[1].data_ptr(), None, None, ctypes.byref(CDisparityWindows(wmin.data_ptr(), wmax.data_ptr(), 3)),
                                       st) == -1
    try:
        lb.set_search_engine("tensor")
        assert call(good) == -2 and "tensor-core" in L.bicos_b200_last_error().decode()
        with pytest.raises(lb.BicosError, match="tensor-core"):
            handle.search(d, d, 4, cols, FLAG_NODUPES, windows=(wmin, wmax))
    finally:
        lb.set_search_engine("auto")
    for margin, fb in ((-1, None), (32768, None), (0, (0, 40000))):
        with pytest.raises(lb.BicosError):
            handle.windows_from_disparity(disp, margin, fb)
    assert handle.kernel_launches == before
    handle.match_windows(l, r, (wmin, wmax), Config())  # the handle is still usable
    assert handle.kernel_launches == before + 4  # two transforms, one search, one refine
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, no_dupes=True, double=True),
                                dict(nxcorr_threshold=None, consistency=True)])
def test_windows_kernels_write_only_their_buffers(handle, kw):
    """Guard words around the key arrays of the stage and the outputs of the match: intact guards, full interiors."""
    import torch

    from libbicos_b200 import capi

    L = lb.lib()
    rows, cols, n = 9, 301, 33
    cfg = Config(**kw)
    ccfg = cfg.to_c()
    left, right, _ = synth.make_stacks(n, 64, cols, np.uint8, seed=5, rows=rows)
    l, r = _cuda(left), _cuda(right)
    p0, _, _, _, pitch, depth = handle._stack_info(l)
    p1 = handle._stack_info(r)[0]
    rng = np.random.default_rng(1)
    wmin, wmax = make_windows("partly_empty", rows, cols, rng)
    maps = _maps(wmin, wmax)  # kept alive while the kernels read them
    win = capi.CDisparityWindows(maps[0].data_ptr(), maps[1].data_ptr(), cols * 2)
    k = lb.descriptor_words(n)
    pw = (cols * k + 3) // 4 * 4
    GUARD, MARK = 1024, 0x5A5A5A5A

    def guarded(words):
        buf = torch.full((GUARD + words + GUARD,), MARK, dtype=torch.int32, device="cuda")
        return buf, buf.data_ptr() + 4 * GUARD

    def intact(buf, words, what, filled=True):
        assert bool((buf[:GUARD] == MARK).all()) and bool((buf[GUARD + words:] == MARK).all()), f"{what}: guard overwritten"
        if filled:
            assert int((buf[GUARD:GUARD + words] == MARK).sum()) == 0, f"{what}: interior not completely written"

    st = handle._stream()
    d = [guarded(rows * pw) for _ in range(2)]
    for planes, (_, ptr) in zip((p0, p1), d):
        capi._check(L.bicos_b200_transform(handle._h, planes, n, rows, cols, pitch, depth, 0, ptr, pw, st))
    px = rows * cols
    keys = [guarded(px) for _ in range(4)]
    flags = cfg.flags
    ptrs = [keys[0][1], keys[1][1], keys[2][1] if flags & 2 else None, keys[3][1] if flags == 3 else None]
    capi._check(L.bicos_b200_search_windows(handle._h, d[0][1], d[1][1], k, rows, cols, pw, flags, *ptrs, ctypes.byref(win), st))
    thr = cfg.nxcorr_threshold is not None
    disp_words = px if thr else (px + 1) // 2
    corr_words = px * (2 if cfg.double else 1)
    disp, corr = guarded(disp_words), guarded(corr_words)
    capi._check(L.bicos_b200_match_windows(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), ctypes.byref(win),
                                           disp[1], cols * (4 if thr else 2), corr[1] if thr else None, cols * (8 if cfg.double else 4), st))
    torch.cuda.synchronize()
    for (buf, _), ptr, what in zip(keys, ptrs, NAMES):
        intact(buf, px, what, filled=ptr is not None)
    intact(disp[0], disp_words, "disparity", filled=thr or px % 2 == 0)
    intact(corr[0], corr_words, "corrmap", filled=thr)
    want = window_keys(desc_cost(*(np.asarray(t[0][GUARD:GUARD + rows * pw].cpu().numpy().view(np.uint32)).reshape(rows, pw)[:, :cols * k]
                                   .reshape(rows, cols, k) for t in d)), rows, cols, wmin, wmax, flags)
    got = {name: (buf[GUARD:GUARD + px].cpu().numpy().view(np.uint32).reshape(rows, cols) if ptr is not None else None)
           for (buf, _), ptr, name in zip(keys, ptrs, NAMES)}
    _assert_keys(got, want, "guarded stage")


@pytest.mark.gpu
def test_windows_on_two_streams(handle):
    import torch

    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True)
    left, right, truth = synth.make_stacks(33, 512, 512, np.uint8, seed=7, row0=100, rows=160)
    l, r = _cuda(left), _cuda(right)
    wins = [_maps(*windows_restated(truth.astype(np.float32), m)) for m in (2, 6)]
    want = [tuple(t.clone() for t in handle.match_windows(l, r, w, Config(**kw))) for w in wins]
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    for _ in range(3):
        for s, w in zip((s1, s2), wins):
            with torch.cuda.stream(s):
                outs.append(handle.match_windows(l, r, w, Config(**kw)))
    torch.cuda.synchronize()
    for m, (d, c) in enumerate(outs):
        wd, wc = want[m % 2]
        assert torch.equal(d.isnan(), wd.isnan()) and torch.equal(d.nan_to_num(7.0), wd.nan_to_num(7.0))
        assert torch.equal(c.nan_to_num(7.0), wc.nan_to_num(7.0))


@pytest.mark.gpu
def test_cpp_windows_consumer(tmp_path, handle):
    import torch

    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
    left, right, _ = synth.make_stacks(33, 256, 272, np.uint8, seed=9, row0=64, rows=45)
    _write_input(tmp_path / "in.bin", left, right, kw)
    exe = os.path.join(ROOT, "tests", "cpp", "build", "windows_check")
    res = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), "3"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    got_d, got_c = _read_output(tmp_path / "out.bin")
    l, r = _cuda(left), _cuda(right)
    prior, _ = handle.match(l, r, Config(**kw))
    want_d, want_c = handle.match_windows(l, r, handle.windows_from_disparity(prior, 3), Config(**kw))
    torch.cuda.synchronize()
    assert np.array_equal(got_d, want_d.cpu().numpy(), equal_nan=True) and np.array_equal(got_c, want_c.cpu().numpy(), equal_nan=True)


def _write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]))
        f.write(np.ascontiguousarray(img).tobytes())


def _read_tiff(path):
    """The single-strip little-endian TIFF bicos-cli writes: (int16 or float32 array)."""
    import struct

    raw = open(path, "rb").read()
    assert raw[:4] == b"II*\x00"
    ifd = struct.unpack_from("<I", raw, 4)[0]
    tags = {}
    for e in range(struct.unpack_from("<H", raw, ifd)[0]):
        tag, typ, _, val = struct.unpack_from("<HHII", raw, ifd + 2 + 12 * e)
        tags[tag] = val & 0xFFFF if typ == 3 else val
    dtype = {(16, 2): np.int16, (32, 3): np.float32}[(tags[258], tags[339])]
    rows, cols = tags[257], tags[256]
    return np.frombuffer(raw, dtype=dtype, count=rows * cols, offset=tags[273]).reshape(rows, cols)


@pytest.mark.gpu
@pytest.mark.parametrize("extra,threshold", [([], "0.9"), (["--disparity-range", "10:60"], "0.9"), ([], "0")])
def test_cli_disparity_prior(tmp_path, handle, extra, threshold):
    left, right, _ = synth.make_stacks(20, 256, 208, np.uint8, seed=17, row0=100, rows=40)
    folder = tmp_path / "in"
    folder.mkdir()
    for t in range(left.shape[0]):
        _write_pgm(folder / f"{t}_left.pgm", left[t])
        _write_pgm(folder / f"{t}_right.pgm", right[t])
    cli = os.path.join(ROOT, "libbicos_b200", "bin", "bicos-cli")
    base = [cli, str(folder), "-t", threshold, "-v", "2.0", "--limited"]
    first = subprocess.run(base + ["-o", str(tmp_path / "a.png")], capture_output=True, text=True, timeout=300)
    assert first.returncode == 0, first.stderr
    second = subprocess.run(base + ["-o", str(tmp_path / "b.png"), "--disparity-prior", f"{tmp_path / 'a.tiff'}:3"] + extra,
                            capture_output=True, text=True, timeout=300)
    assert second.returncode == 0, second.stderr
    # the same through the Python API, from the prior as the CLI wrote it (invalid pixels as NaN or -32768)
    thr = float(threshold)
    cfg = Config(nxcorr_threshold=thr if thr > 0 else None, min_variance=2.0)
    prior = _cuda(_read_tiff(tmp_path / "a.tiff").copy())
    fallback = (10, 60) if extra else None
    want, _ = handle.match_windows(_cuda(left), _cuda(right), handle.windows_from_disparity(prior, 3, fallback), cfg)
    want = want.cpu().numpy()
    if want.dtype == np.float32:
        want = np.where(want == -32768.0, np.float32(np.nan), want)  # the CLI masks -32768.0 like NaN
    got = _read_tiff(tmp_path / "b.tiff")
    assert got.tobytes() == want.tobytes()
    bad = subprocess.run(base + ["--disparity-prior", str(tmp_path / "a.tiff")], capture_output=True, text=True, timeout=60)
    assert bad.returncode != 0 and "FILE:MARGIN" in bad.stderr
    small = tmp_path / "small.tiff"
    data = np.zeros((5, 7), np.float32)
    import struct

    entries = [(256, 3, 1, 7), (257, 3, 1, 5), (258, 3, 1, 32), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, 8),
               (277, 3, 1, 1), (278, 3, 1, 5), (279, 4, 1, data.nbytes), (339, 3, 1, 3)]
    ifd = 8 + data.nbytes
    with open(small, "wb") as f:
        f.write(b"II*\x00" + struct.pack("<I", ifd) + data.tobytes() + struct.pack("<H", len(entries)))
        for e in entries:
            f.write(struct.pack("<HHII", *e))
        f.write(struct.pack("<I", 0))
    bad = subprocess.run(base + ["--disparity-prior", f"{small}:2"], capture_output=True, text=True, timeout=60)
    assert bad.returncode != 0 and "7x5" in bad.stderr
