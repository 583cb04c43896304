"""Config::disparity_range: the search over min <= x_left - x_right <= max only.

The reference for the ranged search is _bicos_range below: the oracle's search + postfilter (oracle.port.bicos, the
reference's bicos()) restated over the clipped window, vectorised per disparity. Whole matches compose it with the
oracle's own descriptor transform and refinement (_match_ranged), as the reference's match_impl composes its stages.
CPU: _bicos_range against a brute force over the full cost matrix, and against oracle.port.bicos for a range that covers
the row. GPU: the windowed search kernel through every layer (stage entry point, whole path, batch / rows / host entry
points, C++ API, CLI) against that reference and against the single ranged match.
"""

import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAG_NODUPES, FLAG_CONSISTENCY = 1, 2
FLAGS = [FLAG_NODUPES, FLAG_CONSISTENCY, FLAG_NODUPES | FLAG_CONSISTENCY]
INVALID = -32768


def _random_desc(rng, rows, cols, k, bits):
    """Descriptors with few distinct values per word, so ties and duplicates are frequent."""
    return rng.integers(0, 1 << bits, size=(rows, cols, k), dtype=np.int64).astype(np.uint32)


def _brute(d0, d1, flags, max_lr, lo, hi):
    """The ranged search + postfilter, written out over the full cost matrix of each row."""
    rows, cols, _ = d0.shape
    nodupes = bool(flags & FLAG_NODUPES)
    i = np.arange(cols)[:, None]
    j = np.arange(cols)[None, :]
    inr = (i - j >= lo) & (i - j <= hi)  # [left, right]
    out = np.full((rows, cols), INVALID, dtype=np.int16)

    def first_min(costs, mask):
        if not mask.any():
            return None
        c = np.where(mask, costs, np.iinfo(np.int64).max)
        m = c.min()
        at = np.flatnonzero(c == m)
        return None if nodupes and len(at) > 1 else int(at[0])

    for r in range(rows):
        x = d0[r][:, None, :] ^ d1[r][None, :, :]
        cost = np.unpackbits(x.view(np.uint8), axis=-1).sum(axis=-1).astype(np.int64)  # [left, right]
        for c0 in range(cols):
            best = first_min(cost[c0], inr[c0])
            if best is None:
                continue
            if flags & FLAG_CONSISTENCY:
                rev = first_min(cost[:, best], inr[:, best])
                if rev is None or abs(c0 - rev) > max_lr:
                    continue
                out[r, c0] = (c0 + rev) // 2 - best
            else:
                out[r, c0] = c0 - best
    return out


def _bicos_range(d0, d1, flags, max_lr, lo, hi):
    """bicos() over the window: forward search of left column i over right columns [i - hi, i - lo], reverse search of
    right column b over left columns [b + lo, b + hi], both clipped to the row; first strict minimum, with no-dupes a
    second minimum invalidates; an empty window is invalid. [H, W, K] uint32 descriptors -> int16 [H, W]."""
    if lo > hi:
        raise ValueError("disparity range: min > max")
    rows, cols, _ = d0.shape
    lo, hi = (min(max(v, -cols), cols) for v in (lo, hi))  # i - j lies in [-(cols - 1), cols - 1]: the same pairs
    nodupes = bool(flags & FLAG_NODUPES)
    ds = np.arange(lo, hi + 1)
    dd = np.arange(len(ds))[:, None]
    x = np.arange(cols)
    j = x[None, :] - ds[:, None]  # [D, W]: right column of left pixel x at disparity d
    ib = x[None, :] + ds[:, None]  # [D, W]: left column of right pixel x at disparity d
    big = np.iinfo(np.int64).max
    out = np.full((rows, cols), INVALID, dtype=np.int16)
    for r in range(rows):
        cost = np.bitwise_count(d0[r][None, :, :] ^ d1[r][np.clip(j, 0, cols - 1)]).sum(axis=-1, dtype=np.int64)
        cost = np.where((j >= 0) & (j < cols), cost, big)  # [D, W]: cost of (left x, right x - d)
        fmin = cost.min(axis=0)
        at = cost == fmin
        best = x - ds[len(ds) - 1 - np.argmax(at[::-1], axis=0)]  # lowest right column = largest disparity
        fok = (fmin < big) & ~(nodupes & (at.sum(axis=0) > 1))
        if not flags & FLAG_CONSISTENCY:
            out[r, fok] = (x - best)[fok]
            continue
        rc = np.where((ib >= 0) & (ib < cols), cost[dd, np.clip(ib, 0, cols - 1)], big)  # [D, W]: (left x + d, right x)
        rmin = rc.min(axis=0)
        rat = rc == rmin
        rev = x + ds[np.argmax(rat, axis=0)]  # lowest left column = smallest disparity
        rok = (rmin < big) & ~(nodupes & (rat.sum(axis=0) > 1))
        b = np.clip(best, 0, cols - 1)
        ok = fok & rok[b] & (np.abs(x - rev[b]) <= max_lr)
        out[r, ok] = ((x + rev[b]) // 2 - best)[ok]
    return out


def _match_ranged(oracles, left, right, drange, nxcorr_threshold=0.5, subpixel_step=None, min_variance=None, mode_full=False,
                  consistency=False, max_lr_diff=1, no_dupes=False, double=False):
    """A ranged BICOS::match from the oracle's stages: descriptors -> _bicos_range -> agree (match_impl's sequence)."""
    port = oracles.port
    d0, d1 = port.descriptors(left, mode_full), port.descriptors(right, mode_full)
    flags = (FLAG_CONSISTENCY | (FLAG_NODUPES if no_dupes else 0)) if consistency else FLAG_NODUPES
    raw = _bicos_range(d0, d1, flags, max_lr_diff if consistency else -1, *drange)
    if nxcorr_threshold is None:
        return raw, None
    disp, corr = port.agree(raw, left, right, nxcorr_threshold, subpixel_step, min_variance, double=double)
    return (disp.astype(np.float32) if subpixel_step is None else disp), corr  # integer mode keeps -32768 as -32768.0f


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)


RANGES_CPU = [(0, 10), (-5, 5), (3, 3), (-20, -3), (60, 70), (-200, -190), (-1000, 1000), (38, 200)]


@pytest.mark.parametrize("k", [1, 2, 4])
@pytest.mark.parametrize("flags", FLAGS)
def test_windowed_reference_equals_brute_force(k, flags):
    rng = np.random.default_rng(10 * k + flags)
    rows, cols = 3, 40  # ranges reach outside the image on both sides and past the row's width
    d0 = _random_desc(rng, rows, cols, k, 2)
    d1 = _random_desc(rng, rows, cols, k, 2)
    d0[:, 10:30] = d1[:, 4:24]  # some unique matches at disparity 6
    for lo, hi in RANGES_CPU:
        want = _brute(d0, d1, flags, 2, lo, hi)
        got = _bicos_range(d0, d1, flags, 2, lo, hi)
        assert np.array_equal(got, want), (lo, hi, int((got != want).sum()))


@pytest.mark.parametrize("flags", FLAGS)
def test_covering_range_equals_the_oracle_full_row(oracles, flags):
    rng = np.random.default_rng(flags)
    rows, cols = 4, 90
    d0 = _random_desc(rng, rows, cols, 2, 3)
    d1 = _random_desc(rng, rows, cols, 2, 3)
    want = oracles.port.bicos(d0, d1, flags, 1)
    for rng_ in ((-(cols - 1), cols - 1), (-cols, cols), (-100000, 100000)):
        assert np.array_equal(_bicos_range(d0, d1, flags, 1, *rng_), want)
    with pytest.raises(ValueError, match="min > max"):
        _bicos_range(d0, d1, flags, 1, 3, 2)


@pytest.mark.parametrize("kw", [dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2, no_dupes=True),
                                dict(nxcorr_threshold=0.8, min_variance=1.0), dict(nxcorr_threshold=None)])
def test_ranged_match_reference_with_a_covering_range_is_the_oracle_match(oracles, kw):
    left, right, _ = synth.make_stacks(17, 256, 120, np.uint8, seed=2, row0=40, rows=12)
    want = oracles.port.match(left, right, **kw)
    got = _match_ranged(oracles, left, right, (-120, 120), **kw)
    assert _same(got[0], want[0]) and ((got[1] is None and want[1] is None) or _same(got[1], want[1]))


def test_config_carries_the_range_to_the_c_struct():
    c = Config(disparity_range=(-7, 12)).to_c()
    assert (c.has_disparity_range, c.min_disparity, c.max_disparity) == (1, -7, 12)
    assert Config().to_c().has_disparity_range == 0
    assert ctypes.sizeof(c) == 4 * 13


def test_range_check_binary_is_built():
    assert os.path.exists(os.path.join(ROOT, "tests", "cpp", "build", "range_check"))


# ------------------------------------------------------------------------------- GPU --
def _cuda(a):
    import torch

    if a.dtype == np.uint16:
        return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(a).cuda()


def _pitched(d):
    import torch

    rows, cols, k = d.shape
    buf = np.zeros((rows, (cols * k + 3) // 4 * 4), dtype=np.uint32)
    buf[:, : cols * k] = d.reshape(rows, cols * k)
    return torch.from_numpy(buf.view(np.int32)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 4, 8, 12, 16])
@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("cols,bits", [(97, 3), (700, 32), (1300, 5), (9000, 4)])
def test_search_range_stage_bit_exact(handle, k, flags, cols, bits):
    import torch

    rng = np.random.default_rng(k * 100 + flags * 10 + cols)
    rows = 4
    d0 = _random_desc(rng, rows, cols, k, bits)
    d1 = _random_desc(rng, rows, cols, k, bits)
    src = rng.integers(0, cols, size=cols // 2)
    dst = np.clip(src + rng.integers(-30, 70, size=cols // 2), 0, cols - 1)
    d0[:, dst] = d1[:, src] ^ (rng.integers(0, 2, size=(rows, cols // 2, k)) << 7).astype(np.uint32)
    max_lr = 3
    dummy = torch.zeros((2, rows, cols), dtype=torch.uint8, device="cuda")
    p0, p1 = _pitched(d0), _pitched(d1)
    for lo, hi in ((0, 63), (-20, 40), (5, 5), (-3000, -2990), (cols + 3, cols + 50)):  # the last: empty for every pixel
        want = _bicos_range(d0, d1, flags, max_lr, lo, hi)
        keys = handle.search(p0, p1, k, cols, flags, disparity_range=(lo, hi))
        assert lb.last_search_kernel() == f"range<K={k},flags={flags}>"
        cfg = Config(nxcorr_threshold=None, consistency=bool(flags & FLAG_CONSISTENCY), max_lr_diff=max_lr,
                     no_dupes=flags == 3, disparity_range=(lo, hi))
        disp, corr, raw = handle.refine(dummy, dummy, cfg, keys)
        got = disp.cpu().numpy()
        assert np.array_equal(got, want), f"range {lo}..{hi}: {(got != want).sum()} of {got.size} differ"
        assert np.array_equal(raw.cpu().numpy(), want)
        if lo > cols:
            assert (got == INVALID).all()


CASES = [
    # n, dtype, rows, cols, config (the whole-path shapes and configurations of test_gpu_parity.py)
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0)),
    (33, np.uint8, 48, 320, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=None)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2, no_dupes=True)),
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, min_variance=1.0)),
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, subpixel_step=0.1, consistency=True)),
    (64, np.uint8, 32, 256, dict(nxcorr_threshold=0.9, subpixel_step=0.2, min_variance=2.0)),
    (9, np.uint8, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.3)),
    (17, np.uint16, 32, 200, dict(nxcorr_threshold=0.8, subpixel_step=0.15, min_variance=4.0)),
    (12, np.uint8, 32, 200, dict(nxcorr_threshold=0.7, mode_full=True, consistency=True, max_lr_diff=0)),
    (5, np.uint16, 16, 101, dict(nxcorr_threshold=0.5, min_variance=0.0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,rows,cols,kw", CASES)
@pytest.mark.parametrize("drange", [(10, 90), (-8, 40)])  # the scene's disparities are 17..75 px
@pytest.mark.parametrize("double", [False, True])
def test_ranged_match_parity(handle, oracles, n, dtype, rows, cols, kw, drange, double):
    if double and kw["nxcorr_threshold"] is None:
        pytest.skip("no correlation stage, no precision")
    left, right, _ = synth.make_stacks(n, 512, cols, dtype, seed=11 * n + cols, row0=128, rows=rows)
    want_d, want_c = _match_ranged(oracles, left, right, drange, double=double, **kw)
    disp, corr = handle.match(_cuda(left), _cuda(right), Config(double=double, disparity_range=drange, **kw))
    assert lb.last_search_kernel().startswith("range<")
    got_d = disp.cpu().numpy()
    assert got_d.dtype == want_d.dtype
    if want_d.dtype == np.int16:
        assert np.array_equal(got_d, want_d) and corr is None
        return
    got_c = corr.cpu().numpy()
    invalid_w = np.isnan(want_d) | (want_d == -32768)
    invalid_g = np.isnan(got_d) | (got_d == -32768)
    edge = np.abs(np.nan_to_num(want_c, nan=9.0) - kw["nxcorr_threshold"]) < 1e-6
    assert np.array_equal(invalid_g | edge, invalid_w | edge), "valid masks differ"
    assert np.array_equal(np.isnan(got_c), np.isnan(want_c))
    ok = ~np.isnan(want_c)
    assert np.max(np.abs(got_c[ok] - want_c[ok]), initial=0) <= (1e-12 if double else 1e-5)
    both = ~(invalid_w | invalid_g)
    assert np.max(np.abs(got_d[both] - want_d[both]), initial=0) <= 1e-3
    if not double:
        assert _same(got_c, want_c) and _same(got_d, want_d)
    if not kw.get("consistency"):  # integer disparities stay inside the range, subpixel ones within 1 px of it
        slack = 0 if kw.get("subpixel_step") is None else 1
        assert ((got_d[both] >= drange[0] - slack) & (got_d[both] <= drange[1] + slack)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,rows,cols,kw", [
    (33, np.uint8, 160, 512, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (33, np.uint8, 40, 300, dict(nxcorr_threshold=None)),
    (16, np.uint16, 40, 288, dict(nxcorr_threshold=0.9, mode_full=True, consistency=True, no_dupes=True)),
])
def test_covering_range_is_the_unranged_match(handle, n, dtype, rows, cols, kw):
    left, right, _ = synth.make_stacks(n, 1024, cols, dtype, seed=n + cols, row0=300, rows=rows)
    l, r = _cuda(left), _cuda(right)
    want_d, want_c = handle.match(l, r, Config(**kw))
    kernel = lb.last_search_kernel()
    assert not kernel.startswith("range<")
    for drange in ((-(cols - 1), cols - 1), (-cols, cols), (-40000, 40000)):
        got_d, got_c = handle.match(l, r, Config(disparity_range=drange, **kw))
        assert lb.last_search_kernel() == kernel
        assert _same(got_d.cpu().numpy(), want_d.cpu().numpy())
        assert (got_c is None) == (want_c is None)
        if got_c is not None:
            assert _same(got_c.cpu().numpy(), want_c.cpu().numpy())


@pytest.mark.gpu
def test_ranged_entry_points_equal_the_single_match(handle):
    import torch

    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1,
              disparity_range=(10, 90))
    cfg = Config(**kw)
    host = [synth.make_stacks(33, 1024, 512, np.uint8, seed=31, frame=f, row0=200, rows=160)[:2] for f in range(3)]
    frames = [(_cuda(a), _cuda(b)) for a, b in host]
    single = [tuple(t.cpu().numpy() for t in handle.match(a, b, cfg)) for a, b in frames]
    assert lb.last_search_kernel() == "range<K=4,flags=2>"

    def check(got, want):
        assert _same(np.asarray(got[0]), want[0]) and _same(np.asarray(got[1]), want[1])

    for overlap in (True, False):
        handle.set_overlap(overlap)
        try:
            for (d, c), want in zip(handle.match_batch(frames, cfg), single):
                check((d.cpu().numpy(), c.cpu().numpy()), want)
            d, c = handle.match(*frames[0], cfg)
            check((d.cpu().numpy(), c.cpu().numpy()), single[0])
        finally:
            handle.set_overlap(True)
    disp = torch.full((160, 512), 7.0, dtype=torch.float32, device="cuda")
    corr = torch.full((160, 512), 7.0, dtype=torch.float32, device="cuda")
    for rb, re in ((0, 50), (50, 111), (111, 160)):
        handle.match(*frames[1], cfg, out=(disp, corr), rows_range=(rb, re))
    check((disp.cpu().numpy(), corr.cpu().numpy()), single[1])
    check(handle.match_host(*host[2], cfg), single[2])
    other = lb.Handle(0)
    try:
        got = [h.match_host_begin(*host[f], cfg) for f, h in ((0, handle), (1, other))]
        handle.match_host_end()
        other.match_host_end()
        for g, want in zip(got, single[:2]):
            check(g, want)
    finally:
        other.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,rows,cols,kw,drange", [
    (33, np.uint8, 7, 300, dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=1, no_dupes=True), (-5, 60)),
    (33, np.uint8, 9, 513, dict(nxcorr_threshold=0.9, subpixel_step=0.5, consistency=True), (0, 400)),
    (16, np.uint16, 5, 131, dict(nxcorr_threshold=0.9, mode_full=True, double=True, min_variance=1.0), (3, 3)),
    (9, np.uint8, 3, 1, dict(nxcorr_threshold=None), (1, 1)),  # one column: (0, 0) would cover the row, (1, 1) is empty
    (9, np.uint8, 6, 200, dict(nxcorr_threshold=None), (250, 300)),  # empty for every pixel
])
def test_range_kernel_writes_only_its_buffers(handle, n, dtype, rows, cols, kw, drange):
    """Guard words around every buffer of the ranged stages and the ranged match (test_kernels_write_only_their_buffers
    for the windowed search): intact guards, completely written interiors."""
    import torch

    from libbicos_b200 import capi

    L = lb.lib()
    cfg = Config(disparity_range=drange, **kw)
    ccfg = cfg.to_c()
    full = kw.get("mode_full", False)
    left, right, _ = synth.make_stacks(n, 64, max(cols, 16), dtype, seed=n + cols, rows=rows)
    l, r = _cuda(np.ascontiguousarray(left[:, :, :cols])), _cuda(np.ascontiguousarray(right[:, :, :cols]))
    p0, _, _, _, pitch, depth = handle._stack_info(l)
    p1 = handle._stack_info(r)[0]
    k = lb.descriptor_words(n, full)
    pw = (cols * k + 3) // 4 * 4
    GUARD, MARK = 1024, 0x5A5A5A5A

    def guarded(words):
        buf = torch.full((GUARD + words + GUARD,), MARK, dtype=torch.int32, device="cuda")
        return buf, buf.data_ptr() + 4 * GUARD

    def intact(buf, words, what, filled=True):
        assert bool((buf[:GUARD] == MARK).all()) and bool((buf[GUARD + words:] == MARK).all()), f"{what}: guard words overwritten"
        if filled:
            assert int((buf[GUARD : GUARD + words] == MARK).sum()) == 0, f"{what}: interior not completely written"

    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    px = rows * cols
    d = [guarded(rows * pw) for _ in range(2)]
    for planes, (_, ptr) in zip((p0, p1), d):
        capi._check(L.bicos_b200_transform(handle._h, planes, n, rows, cols, pitch, depth, int(full), ptr, pw, st))
    keys = [guarded(px) for _ in range(4)]
    flags = cfg.flags
    ptrs = [keys[0][1], keys[1][1], keys[2][1] if flags & 2 else None, keys[3][1] if flags == 3 else None]
    capi._check(L.bicos_b200_search_range(handle._h, d[0][1], d[1][1], k, rows, cols, pw, flags, *ptrs, drange[0], drange[1], st))
    assert lb.last_search_kernel().startswith("range<")
    thr = cfg.nxcorr_threshold is not None
    disp_words = px if thr else (px + 1) // 2
    corr_words = px * (2 if cfg.double else 1)
    raw, disp, corr = guarded((px + 1) // 2), guarded(disp_words), guarded(corr_words)
    disp_pitch = cols * (4 if thr else 2)
    capi._check(L.bicos_b200_refine(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), *ptrs, raw[1], disp[1],
                                    disp_pitch, corr[1] if thr else None, cols * (8 if cfg.double else 4), st))
    torch.cuda.synchronize()
    odd = px % 2 == 1
    for (buf, _), what in zip(d, ("desc0", "desc1")):
        intact(buf, rows * pw, what, filled=pw == cols * k)
    for (buf, _), ptr, what in zip(keys, ptrs, ("fwd_first", "fwd_last", "rev_first", "rev_last")):
        intact(buf, px, what, filled=ptr is not None)
    intact(raw[0], (px + 1) // 2, "raw disparity", filled=not odd)
    intact(disp[0], disp_words, "disparity", filled=thr or not odd)
    intact(corr[0], corr_words, "corrmap", filled=thr)
    disp2, corr2 = guarded(disp_words), guarded(corr_words)
    capi._check(L.bicos_b200_match(handle._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), disp2[1], disp_pitch,
                                   corr2[1] if thr else None, cols * (8 if cfg.double else 4), st))
    torch.cuda.synchronize()
    intact(disp2[0], disp_words, "match disparity", filled=thr or not odd)
    intact(corr2[0], corr_words, "match corrmap", filled=thr)
    assert torch.equal(disp2[0], disp[0]) and torch.equal(corr2[0], corr[0])


@pytest.mark.gpu
def test_range_errors(handle):
    import torch

    left, right, _ = synth.make_stacks(9, 32, 64, np.uint8, seed=3)
    l, r = _cuda(left), _cuda(right)
    with pytest.raises(lb.BicosError, match="min > max"):
        handle.match(l, r, Config(disparity_range=(5, 4)))
    with pytest.raises(lb.BicosError, match="min > max"):
        handle.match_host(left, right, Config(disparity_range=(0, -1)))
    d = torch.zeros((2, 64), dtype=torch.int32, device="cuda")
    with pytest.raises(lb.BicosError, match="min > max"):
        handle.search(d, d, 1, 64, FLAG_NODUPES, disparity_range=(1, 0))
    # the tensor-core engine has no windowed kernel: forcing it fails instead of falling back
    try:
        lb.set_search_engine("tensor")
        with pytest.raises(lb.BicosError, match="tensor-core"):
            handle.match(l, r, Config(disparity_range=(0, 20)))
        d4 = torch.zeros((2, 64 * 4), dtype=torch.int32, device="cuda")
        with pytest.raises(lb.BicosError, match="tensor-core"):
            handle.search(d4, d4, 4, 64, FLAG_NODUPES, disparity_range=(0, 20))
    finally:
        lb.set_search_engine("auto")
    handle.match(l, r, Config(disparity_range=(0, 20)))  # the handle is still usable
    torch.cuda.synchronize()


def _write_input(path, left, right, kw):
    """tests/cpp/api_check.cpp's input format."""
    n, rows, cols = left.shape

    def opt(v):
        return -1.0 if v is None else float(v)

    with open(path, "wb") as f:
        f.write(struct.pack("<9i", n, rows, cols, 2 if left.dtype == np.uint16 else 0, int(kw.get("mode_full", False)),
                            int(kw.get("double", False)), int(kw.get("consistency", False)), int(kw.get("max_lr_diff", 1)),
                            int(kw.get("no_dupes", False))))
        f.write(struct.pack("<3f", opt(kw.get("nxcorr_threshold", 0.5)), opt(kw.get("subpixel_step")), opt(kw.get("min_variance"))))
        f.write(np.ascontiguousarray(left).tobytes())
        f.write(np.ascontiguousarray(right).tobytes())


def _read_output(path):
    raw = open(path, "rb").read()
    dt, ct, rows, cols = struct.unpack("<4i", raw[:16])
    types = {3: np.int16, 5: np.float32, 6: np.float64}
    d = np.frombuffer(raw, dtype=types[dt], count=rows * cols, offset=16).reshape(rows, cols)
    c = np.frombuffer(raw, dtype=types[ct], count=rows * cols, offset=16 + d.nbytes).reshape(rows, cols) if ct else None
    return d, c


@pytest.mark.gpu
@pytest.mark.parametrize("sharded", [False, True])
def test_cpp_config_range_reaches_the_kernels(tmp_path, oracles, sharded):
    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
    left, right, _ = synth.make_stacks(33, 256, 272, np.uint8, seed=9, row0=64, rows=45)
    want_d, want_c = _match_ranged(oracles, left, right, (-4, 50), **kw)
    _write_input(tmp_path / "in.bin", left, right, kw)
    exe = os.path.join(ROOT, "tests", "cpp", "build", "range_check")
    res = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), "-4", "50"] + (["sharded"] if sharded else []),
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    got_d, got_c = _read_output(tmp_path / "out.bin")
    assert _same(got_d, want_d) and _same(got_c, want_c)
    unranged = oracles.port.match(left, right, **kw)[0]
    assert not _same(got_d, unranged), "the scene should tell the range from the full row"


@pytest.mark.gpu
def test_cli_disparity_range(tmp_path, handle):
    cv2 = pytest.importorskip("cv2")
    left, right, _ = synth.make_stacks(20, 256, 208, np.uint8, seed=17, row0=100, rows=40)
    folder = tmp_path / "in"
    folder.mkdir()
    for t in range(left.shape[0]):
        assert cv2.imwrite(str(folder / f"{t}_left.png"), left[t])
        assert cv2.imwrite(str(folder / f"{t}_right.png"), right[t])
    out = tmp_path / "disp.png"
    cli = os.path.join(ROOT, "libbicos_b200", "bin", "bicos-cli")
    res = subprocess.run([cli, str(folder), "-o", str(out), "-t", "0.9", "-v", "2.0", "--limited", "--disparity-range", "-5:30"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    want, _ = handle.match_host(left, right, Config(nxcorr_threshold=0.9, min_variance=2.0, disparity_range=(-5, 30)))
    got = cv2.imread(str(tmp_path / "disp.tiff"), cv2.IMREAD_UNCHANGED)
    invalid = np.isnan(want) | (want == -32768)
    assert got is not None and np.array_equal(np.isnan(got), invalid)  # the CLI masks -32768.0 like NaN
    assert np.array_equal(got[~invalid], want[~invalid])
    bad = subprocess.run([cli, str(folder), "--disparity-range", "5"], capture_output=True, text=True, timeout=60)
    assert bad.returncode != 0 and "MIN:MAX" in bad.stderr
