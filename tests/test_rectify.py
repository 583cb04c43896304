"""Rectification on the device: the remap stage (bicos_b200_remap) and match_rectified on raw stacks.

The reference for the stage is _remap below, a numpy restatement of OpenCV's CPU cv::remap(INTER_LINEAR,
BORDER_CONSTANT 0) on float32 maps as include/bicos_b200.h states it. CPU: the restatement against cv2.remap's outputs
stored in tests/golden/remap/remap_cv2.npz (tests/golden/make_remap_golden.py), against live cv2 where it is installed, and on
identity and shift maps. GPU: Handle.remap bit-exact against the restatement and the stored cv2 outputs; match_rectified
bit-identical to match() of the remapped stacks through every path of the match; errors, launch count and the C++ API.
"""

import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config, RectifyMaps, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "remap", "remap_cv2.npz")
MAP_LIMIT = 2.0 ** 25


def _remap(src, mx, my):
    """cv::remap(src, mx, my, INTER_LINEAR, BORDER_CONSTANT, 0) for uint8 / uint16 src [..., H, W] and float32 maps
    [rows, cols] -> [..., rows, cols]: taps at 1/32 px (round half to even), int32 fixed-point weights for 8U, float32
    weights and a left-to-right sum of rounded products for 16U, 0 outside the source and for NaN / inf / |m| >= 2^25."""
    mx = np.asarray(mx, dtype=np.float32)
    my = np.asarray(my, dtype=np.float32)
    ok = (np.abs(mx) < MAP_LIMIT) & (np.abs(my) < MAP_LIMIT)
    X = np.rint(np.where(ok, mx, 0).astype(np.float64) * 32).astype(np.int64)  # m * 32 is exact; rint rounds half to even
    Y = np.rint(np.where(ok, my, 0).astype(np.float64) * 32).astype(np.int64)
    x0, y0, fx, fy = X >> 5, Y >> 5, X & 31, Y & 31
    H, W = src.shape[-2:]

    def tap(yy, xx):
        inside = ok & (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
        return np.where(inside, src[..., np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)], 0).astype(np.int64)

    v00, v01, v10, v11 = tap(y0, x0), tap(y0, x0 + 1), tap(y0 + 1, x0), tap(y0 + 1, x0 + 1)
    if src.dtype == np.uint8:
        return (((32 - fx) * (32 - fy) * v00 + fx * (32 - fy) * v01 + (32 - fx) * fy * v10 + fx * fy * v11 + 512) >> 10).astype(np.uint8)
    f32 = np.float32
    ax, ay = fx.astype(f32) * f32(1 / 32), fy.astype(f32) * f32(1 / 32)
    one = f32(1)
    w00, w01, w10, w11 = (one - ay) * (one - ax), (one - ay) * ax, ay * (one - ax), ay * ax
    s = v00.astype(f32) * w00 + v01.astype(f32) * w01  # numpy rounds every float32 product and sum on its own
    s = (s + v10.astype(f32) * w10) + v11.astype(f32) * w11
    return np.clip(np.rint(s), 0, 65535).astype(np.uint16)


def _golden():
    g = np.load(GOLDEN)
    return g, [k[:-3] for k in g.files if k.endswith("_mx")]


@pytest.mark.parametrize("src", ["src8", "src16"])
def test_restatement_equals_stored_cv2(src):
    g, names = _golden()
    assert set(names) == {"random", "ties", "special"}
    for name in names:
        want = g[f"{name}_{src}"]
        got = _remap(g[src], g[f"{name}_mx"], g[f"{name}_my"])
        assert got.dtype == want.dtype and np.array_equal(got, want), f"{name}: {(got != want).sum()} of {got.size} differ"


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_restatement_equals_live_cv2(dtype):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    src = rng.integers(0, np.iinfo(dtype).max + 1, (90, 130), dtype=dtype)
    maps = [synth.rectify_maps(70, 150, 90, 130), synth.rectify_maps(70, 150, 90, 130, camera=1, k1=0.2),
            (rng.uniform(-4, 133, (70, 150)), rng.uniform(-4, 93, (70, 150))),
            (rng.integers(-256, 134 * 64, (70, 150)) / 64.0, rng.integers(-256, 94 * 64, (70, 150)) / 64.0)]
    for mx, my in maps:
        mx, my = mx.astype(np.float32), my.astype(np.float32)
        want = cv2.remap(src, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        assert np.array_equal(_remap(src, mx, my), want)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_restatement_identity_and_shifts(dtype):
    rng = np.random.default_rng(3)
    src = rng.integers(0, np.iinfo(dtype).max + 1, (3, 20, 31), dtype=dtype)
    y, x = np.mgrid[0:20, 0:31].astype(np.float32)
    assert np.array_equal(_remap(src, x, y), src)
    for dy, dx in ((0, 3), (2, -5), (-1, 0), (-7, 11)):
        want = np.zeros_like(src)
        for yy in range(20):
            for xx in range(31):
                if 0 <= yy + dy < 20 and 0 <= xx + dx < 31:
                    want[:, yy, xx] = src[:, yy + dy, xx + dx]
        assert np.array_equal(_remap(src, x + dx, y + dy), want), (dy, dx)


def test_rectify_maps_struct_layout():
    assert ctypes.sizeof(lb.capi.CRectifyMaps) == 5 * 8
    assert {"bicos_b200_remap", "bicos_b200_match_rectified"} <= set(lb.capi.EXPORTS)


def test_rectify_check_binary_is_built():
    assert os.path.exists(os.path.join(ROOT, "tests", "cpp", "build", "rectify_check"))


# ------------------------------------------------------------------------------- GPU --
def _cuda(a):
    import torch

    if a.dtype == np.uint16:
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    import torch

    if t.dtype == torch.uint16:
        return t.view(torch.int16).cpu().numpy().view(np.uint16)
    return t.cpu().numpy()


def _padded(a, pad):
    """A CUDA view of `a` [..., rows, cols] whose rows lie `pad` elements apart beyond the minimal pitch."""
    import torch

    buf = np.zeros(a.shape[:-1] + (a.shape[-1] + pad,), dtype=a.dtype)
    buf[..., : a.shape[-1]] = a
    t = _cuda(buf) if a.dtype != np.float32 else torch.from_numpy(buf).cuda()
    return t[..., : a.shape[-1]]


def _maps_cuda(mx, my, pad=0):
    return _padded(mx.astype(np.float32), pad), _padded(my.astype(np.float32), pad)


def _wild_maps(rng, rows, cols, src_rows, src_cols):
    """Realistic maps with a quarter of the values replaced by NaN, inf or far-away coordinates."""
    mx, my = synth.rectify_maps(rows, cols, src_rows, src_cols, k1=0.25)
    bad = np.array([np.nan, np.inf, -np.inf, 1e6, -1e6, 3e9, -3e9, 4e7, -0.5, -0.99, -1.02], dtype=np.float32)
    pick = rng.random((rows, cols))
    mx = np.where(pick < 0.15, rng.choice(bad, (rows, cols)), mx)
    my = np.where((pick > 0.1) & (pick < 0.25), rng.choice(bad, (rows, cols)), my)
    return mx.astype(np.float32), my.astype(np.float32)


# source larger than, smaller than and equal to the output; output widths not multiples of 4
SHAPES = [((70, 131), (53, 97)), ((41, 59), (64, 103)), ((48, 90), (48, 90))]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 17, 33, 65])
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
@pytest.mark.parametrize("shape", SHAPES)
def test_remap_stage_bit_exact(handle, n, dtype, shape):
    """Handle.remap against the restatement, with non-minimal source, map and output pitches and guard words around
    every output plane and in its pitch padding."""
    import torch

    (src_rows, src_cols), (rows, cols) = shape
    rng = np.random.default_rng(n * 1000 + src_cols + rows)
    src = rng.integers(0, np.iinfo(dtype).max + 1, (n, src_rows, src_cols), dtype=dtype)
    s = _padded(src, 5)
    PAD, GUARD = 7, 300  # output pitch = cols + 7 elements; GUARD elements before the first and after the last plane
    MARK = 0xA5 if dtype == np.uint8 else 0xA5A5
    for maps in (synth.rectify_maps(rows, cols, src_rows, src_cols), _wild_maps(rng, rows, cols, src_rows, src_cols),
                 (rng.uniform(-3, src_cols + 2, (rows, cols)), rng.uniform(-3, src_rows + 2, (rows, cols)))):
        mx, my = maps
        want = _remap(src, mx, my)
        flat = _cuda(np.full(GUARD + n * rows * (cols + PAD) + GUARD, MARK, dtype=dtype))
        out = flat[GUARD:-GUARD].view(n, rows, cols + PAD)[:, :, :cols]
        got = handle.remap(s, *_maps_cuda(mx, my, pad=3), out=out)
        assert got.data_ptr() == out.data_ptr()
        torch.cuda.synchronize()
        assert np.array_equal(_np(got), want), f"{(_np(got) != want).sum()} of {want.size} differ"
        f = _np(flat)
        assert (f[:GUARD] == MARK).all() and (f[-GUARD:] == MARK).all(), "guard words around the planes overwritten"
        assert (f[GUARD:-GUARD].reshape(n, rows, cols + PAD)[:, :, cols:] == MARK).all(), "pitch padding overwritten"
        dense = handle.remap(_cuda(src), *_maps_cuda(mx, my))
        assert np.array_equal(_np(dense), want)


@pytest.mark.gpu
@pytest.mark.parametrize("src", ["src8", "src16"])
def test_remap_stage_equals_stored_cv2(handle, src):
    g, names = _golden()
    for name in names:
        s = np.repeat(g[src][None], 3, axis=0)
        got = _np(handle.remap(_cuda(s), *_maps_cuda(g[f"{name}_mx"], g[f"{name}_my"])))
        assert np.array_equal(got, np.repeat(g[f"{name}_{src}"][None], 3, axis=0)), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_remap_identity_maps_reproduce_the_input(handle, dtype):
    left, _, _ = synth.make_stacks(9, 64, 203, dtype, seed=5)
    y, x = np.mgrid[0:64, 0:203].astype(np.float32)
    assert np.array_equal(_np(handle.remap(_cuda(left), *_maps_cuda(x, y))), left)


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)


def _scene(n, dtype, src_rows, src_cols, rows, cols, seed):
    """Raw stacks of the synthetic scene and mildly distorted maps for both cameras."""
    left, right, _ = synth.make_stacks(n, max(512, src_rows), src_cols, dtype, seed=seed, rows=src_rows)
    m0 = synth.rectify_maps(rows, cols, src_rows, src_cols, camera=0, k1=-0.05, k2=0.0, angle_deg=0.1)
    m1 = synth.rectify_maps(rows, cols, src_rows, src_cols, camera=1, k1=-0.04, k2=0.0, angle_deg=0.1)
    return left, right, m0, m1


def _maps(m0, m1):
    (x0, y0), (x1, y1) = _maps_cuda(*m0), _maps_cuda(*m1)
    return RectifyMaps(x0, y0, x1, y1)


MATCH_CASES = [
    # n, dtype, raw (rows, cols), rectified (rows, cols), config
    (33, np.uint8, (60, 330), (48, 320), dict(nxcorr_threshold=0.96, min_variance=2.0)),
    (33, np.uint8, (60, 330), (48, 320), dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (33, np.uint8, (40, 290), (44, 301), dict(nxcorr_threshold=None)),
    (33, np.uint8, (40, 300), (40, 300), dict(nxcorr_threshold=0.9, subpixel_step=0.25, consistency=True, max_lr_diff=2, no_dupes=True)),
    (16, np.uint16, (50, 300), (40, 288), dict(nxcorr_threshold=0.9, mode_full=True, min_variance=1.0)),
    (16, np.uint16, (50, 300), (40, 288), dict(nxcorr_threshold=0.9, mode_full=True, subpixel_step=0.1, consistency=True)),
    (17, np.uint16, (36, 210), (32, 203), dict(nxcorr_threshold=0.8, subpixel_step=0.15, min_variance=4.0)),
    (33, np.uint8, (60, 330), (48, 320), dict(nxcorr_threshold=0.96, subpixel_step=0.1, disparity_range=(10, 90))),
    (16, np.uint16, (50, 300), (40, 288), dict(nxcorr_threshold=0.9, consistency=True, no_dupes=True, disparity_range=(-8, 40))),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,raw,rect,kw", MATCH_CASES)
@pytest.mark.parametrize("double", [False, True])
def test_match_rectified_is_match_of_the_remapped_stacks(handle, n, dtype, raw, rect, kw, double):
    if double and kw["nxcorr_threshold"] is None:
        pytest.skip("no correlation stage, no precision")
    left, right, m0, m1 = _scene(n, dtype, *raw, *rect, seed=n + raw[1])
    cfg = Config(double=double, **kw)
    l, r = _cuda(left), _cuda(right)
    maps = _maps(m0, m1)
    want_d, want_c = handle.match(handle.remap(l, maps.map_x0, maps.map_y0), handle.remap(r, maps.map_x1, maps.map_y1), cfg)
    got_d, got_c = handle.match_rectified(l, r, maps, cfg)
    assert tuple(got_d.shape) == rect
    assert _same(_np(got_d), _np(want_d))
    assert (got_c is None) == (want_c is None)
    if got_c is not None:
        assert _same(_np(got_c), _np(want_c))
        assert np.isfinite(_np(got_c)).mean() > 0.05, "the rectified scene should be evaluated"


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1),
                                dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True)])
@pytest.mark.parametrize("overlap", [True, False])
def test_match_rectified_banded_and_without_overlap(handle, kw, overlap):
    """1536 rectified rows take the row-banded two-stream path of the match (with overlap); the result is the same."""
    left, right, m0, m1 = _scene(33, np.uint8, 1560, 520, 1536, 512, seed=77)
    l, r = _cuda(left), _cuda(right)
    maps = _maps(m0, m1)
    cfg = Config(**kw)
    handle.set_overlap(overlap)
    try:
        want_d, want_c = handle.match(handle.remap(l, maps.map_x0, maps.map_y0), handle.remap(r, maps.map_x1, maps.map_y1), cfg)
        got_d, got_c = handle.match_rectified(l, r, maps, cfg)
        assert _same(_np(got_d), _np(want_d)) and _same(_np(got_c), _np(want_c))
        out = (got_d.clone().fill_(7), got_c.clone().fill_(7))
        handle.match_rectified(l, r, maps, cfg, out=out)
        assert _same(_np(out[0]), _np(want_d)) and _same(_np(out[1]), _np(want_c))
    finally:
        handle.set_overlap(True)


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype,kw", [
    (33, np.uint8, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (16, np.uint16, dict(nxcorr_threshold=0.9, mode_full=True, double=True)),
    (9, np.uint8, dict(nxcorr_threshold=None, consistency=True, no_dupes=True)),
])
def test_identity_maps_make_match_rectified_the_match(handle, n, dtype, kw):
    left, right, _ = synth.make_stacks(n, 512, 301, dtype, seed=n, row0=100, rows=50)
    y, x = np.mgrid[0:50, 0:301].astype(np.float32)
    mx, my = _maps_cuda(x, y)
    l, r = _cuda(left), _cuda(right)
    want_d, want_c = handle.match(l, r, Config(**kw))
    got_d, got_c = handle.match_rectified(l, r, RectifyMaps(mx, my, mx, my), Config(**kw))
    assert _same(_np(got_d), _np(want_d))
    assert (got_c is None) == (want_c is None) and (got_c is None or _same(_np(got_c), _np(want_c)))


@pytest.mark.gpu
def test_match_rectified_equals_the_oracle_on_the_restated_stacks(handle, oracles):
    kw = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
    left, right, m0, m1 = _scene(33, np.uint8, 40, 270, 32, 256, seed=21)
    want_d, want_c = oracles.port.match(_remap(left, *m0), _remap(right, *m1), **kw)
    got_d, got_c = handle.match_rectified(_cuda(left), _cuda(right), _maps(m0, m1), Config(**kw))
    assert _same(_np(got_d), want_d) and _same(_np(got_c), want_c)


@pytest.mark.gpu
def test_one_remap_launch_per_rectified_match(handle):
    left, right, m0, m1 = _scene(17, np.uint8, 50, 200, 40, 192, seed=4)
    l, r = _cuda(left), _cuda(right)
    maps = _maps(m0, m1)
    cfg = Config(nxcorr_threshold=0.9, subpixel_step=0.2)
    rl, rr = handle.remap(l, maps.map_x0, maps.map_y0), handle.remap(r, maps.map_x1, maps.map_y1)
    handle.match(rl, rr, cfg)
    a = handle.kernel_launches
    handle.match(rl, rr, cfg)
    b = handle.kernel_launches
    handle.match_rectified(l, r, maps, cfg)
    c = handle.kernel_launches
    handle.remap(l, maps.map_x0, maps.map_y0)
    assert c - b == (b - a) + 1 and handle.kernel_launches - c == 1


@pytest.mark.gpu
def test_rectify_errors(handle):
    import torch

    from libbicos_b200 import capi

    L = lb.lib()
    left, right, m0, m1 = _scene(9, np.uint8, 40, 100, 32, 96, seed=8)
    l, r = _cuda(left), _cuda(right)
    maps = _maps(m0, m1)
    cfg = Config()
    p0, n, src_rows, src_cols, pitch, depth = handle._stack_info(l)
    p1 = handle._stack_info(r)[0]
    ccfg = cfg.to_c()
    disp = torch.empty((32, 96), dtype=torch.float32, device="cuda")
    corr = torch.empty((32, 96), dtype=torch.float32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    mp = [maps.map_x0.data_ptr(), maps.map_y0.data_ptr(), maps.map_x1.data_ptr(), maps.map_y1.data_ptr()]
    map_pitch = maps.map_x0.stride(0) * 4

    def match_rc(ptrs=mp, pitch_=map_pitch, rows=32, cols=96, depth_=depth, srows=src_rows, scols=src_cols):
        cm = capi.CRectifyMaps(*ptrs, pitch_)
        return L.bicos_b200_match_rectified(handle._h, p0, p1, n, srows, scols, pitch, depth_, ctypes.byref(cm), rows, cols,
                                            ctypes.byref(ccfg), disp.data_ptr(), 96 * 4, corr.data_ptr(), 96 * 4, st)

    before = handle.kernel_launches
    for k in range(4):
        assert match_rc(ptrs=[None if i == k else p for i, p in enumerate(mp)]) == -1
        assert "null" in L.bicos_b200_last_error().decode()
    assert L.bicos_b200_match_rectified(handle._h, p0, p1, n, src_rows, src_cols, pitch, depth, None, 32, 96, ctypes.byref(ccfg),
                                        disp.data_ptr(), 96 * 4, corr.data_ptr(), 96 * 4, st) == -1
    assert match_rc(pitch_=96 * 4 - 4) == -1 and "map" in L.bicos_b200_last_error().decode()
    assert match_rc(pitch_=96 * 4 + 2) == -1
    assert match_rc(depth_=1) == -1 and "depth" in L.bicos_b200_last_error().decode()
    assert match_rc(rows=40000) == -1
    assert match_rc(srows=40000) == -1 and "32767" in L.bicos_b200_last_error().decode()
    assert match_rc(scols=0) == -1
    assert handle.kernel_launches == before, "a rejected call launched something"

    dst = torch.empty((9, 32, 96), dtype=torch.uint8, device="cuda")
    pd = handle._stack_info(dst)[0]

    def remap_rc(mx=mp[0], my=mp[1], pitch_=map_pitch, depth_=depth, dst_pitch=96, n_=n, rows=32, cols=96):
        return L.bicos_b200_remap(handle._h, p0, n_, src_rows, src_cols, pitch, depth_, mx, my, pitch_, rows, cols, pd, dst_pitch, st)

    assert remap_rc() == 0
    for bad in (dict(mx=None), dict(my=None), dict(pitch_=8), dict(pitch_=map_pitch + 1), dict(depth_=5), dict(dst_pitch=95),
                dict(n_=0), dict(n_=66), dict(rows=32768), dict(cols=0)):
        assert remap_rc(**bad) == -1, bad
    with pytest.raises(lb.BicosError, match="float32"):
        handle.remap(l, maps.map_x0.double(), maps.map_y0)
    with pytest.raises(lb.BicosError, match="share one shape"):
        handle.match_rectified(l, r, RectifyMaps(maps.map_x0, maps.map_y0, maps.map_x1, maps.map_y1[:-1]), cfg)
    with pytest.raises(lb.BicosError, match="min > max"):
        handle.match_rectified(l, r, maps, Config(disparity_range=(5, 4)))
    with pytest.raises(lb.BicosError):
        handle.match_rectified(l[:1], r[:1], maps, cfg)  # one image: the match needs two
    handle.match_rectified(l, r, maps, cfg)  # the handle is still usable
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


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,kw", [
    (np.uint8, dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)),
    (np.uint16, dict(nxcorr_threshold=0.9, mode_full=True, double=True)),
])
def test_cpp_match_rectified_and_remap(tmp_path, handle, dtype, kw):
    n = 33 if dtype == np.uint8 else 16
    left, right, m0, m1 = _scene(n, dtype, 50, 280, 45, 272, seed=9)
    _write_input(tmp_path / "in.bin", left, right, kw)
    with open(tmp_path / "maps.bin", "wb") as f:
        f.write(struct.pack("<2i", 45, 272))
        for m in (*m0, *m1):
            f.write(np.ascontiguousarray(m, dtype=np.float32).tobytes())
    exe = os.path.join(ROOT, "tests", "cpp", "build", "rectify_check")
    res = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "maps.bin"), str(tmp_path / "out.bin")],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    dt, ct, rows, cols = struct.unpack("<4i", raw[:16])
    types = {3: np.int16, 5: np.float32, 6: np.float64}
    got_d = np.frombuffer(raw, dtype=types[dt], count=rows * cols, offset=16).reshape(rows, cols)
    off = 16 + got_d.nbytes
    got_c = np.frombuffer(raw, dtype=types[ct], count=rows * cols, offset=off).reshape(rows, cols)
    off += got_c.nbytes
    got_r = np.frombuffer(raw, dtype=dtype, count=n * rows * cols, offset=off).reshape(n, rows, cols)
    want_d, want_c = handle.match_rectified(_cuda(left), _cuda(right), _maps(m0, m1), Config(**kw))
    assert _same(got_d, _np(want_d)) and _same(got_c, _np(want_c))
    assert np.array_equal(got_r, _remap(left, *m0))


def test_match_rectified_takes_opencv_types(tmp_path):
    """-DBICOS_WITH_OPENCV: RectifyMaps holds cv::cuda::GpuMat and match_rectified takes a cv::cuda::Stream& as match
    does. Compile-only, against the stand-in headers of oracle/shim."""
    src = tmp_path / "rectify_opencv.cpp"
    src.write_text("""#include <BICOS/rectify.hpp>
void calls(const std::vector<cv::cuda::GpuMat>& s0, const std::vector<cv::cuda::GpuMat>& s1, const BICOS::RectifyMaps& maps) {
    cv::cuda::GpuMat disparity, corrmap;
    cv::cuda::Stream stream;
    BICOS::match_rectified(s0, s1, maps, disparity);
    BICOS::match_rectified(s0, s1, maps, disparity, BICOS::Config {}, &corrmap, stream);
    BICOS::match_rectified(s0, s1, maps, disparity, BICOS::Config {}, &corrmap, static_cast<void*>(nullptr));
    std::vector<cv::cuda::GpuMat> rectified;
    BICOS::remap(s0, maps.map_x0, maps.map_y0, rectified);
}
""")
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-DBICOS_WITH_OPENCV", "-I" + os.path.join(ROOT, "oracle", "shim"),
           "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include", str(src)]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
