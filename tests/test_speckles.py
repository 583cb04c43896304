"""Speckle removal on the device: bicos_b200_filter_speckles, BICOS::filter_speckles, Handle.filter_speckles and
bicos-cli --speckles.

The reference is _filter below, a restatement of the semantics include/bicos_b200.h states: numpy for the members and
edges, scipy.sparse.csgraph.connected_components for the components. CPU: the restatement against a plain-Python port
of OpenCV's scan-and-BFS filterSpecklesImpl, against cv2.filterSpeckles outputs stored in
tests/golden/speckles/speckles_cv2.npz (tests/golden/make_speckle_golden.py) and against live cv2 where it is
installed; float32 edges built on the rounding of the difference; the OpenCV-types compile check of the header. GPU:
the kernel bit-exact against the restatement, counts included, over shapes, pitches, real matches and adversarial
connectivity; idempotence, launch counts, errors, two streams, the plain-g++ consumer and the CLI.
"""

import ctypes
import os
import re
import struct
import subprocess

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

import libbicos_b200 as lb
from libbicos_b200 import Config, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "libbicos_b200", "bin", "bicos-cli")
CHECK = os.path.join(ROOT, "tests", "cpp", "build", "speckle_check")
GOLDEN = os.path.join(ROOT, "tests", "golden", "speckles", "speckles_cv2.npz")
MARKER = -32768
TILE_W, TILE_H = 128, 16  # speckles.cu's tile: the adversarial scenes cross its edges


def _params(dtype, new_value, max_diff):
    """(new, diff) as the filter uses them: int16 rounds half to even (cvRound), float32 converts."""
    if np.dtype(dtype) == np.int16:
        return int(np.rint(new_value)), int(np.clip(np.rint(max_diff), -65535, 65535))
    return np.float32(new_value), np.float32(max_diff)


def _members(d, new):
    if d.dtype == np.int16:
        return (d != MARKER) & (d != new)
    return ~np.isnan(d) & (d != np.float32(MARKER)) & (d != new)


def _edges(a, b, diff):
    if a.dtype == np.int16:
        return np.abs(a.astype(np.int32) - b.astype(np.int32)) <= diff
    with np.errstate(all="ignore"):
        return np.abs(a - b) <= diff  # float32 difference, rounded to nearest; NaN compares false


def _filter(disp, new_value, max_speckle_size, max_diff):
    """Restatement -> (filtered copy, (pixels set, speckles removed))."""
    d = np.array(disp, copy=True)
    new, diff = _params(d.dtype, new_value, max_diff)
    if max_speckle_size <= 0:
        return d, (0, 0)
    rows, cols = d.shape
    m = _members(d, new)
    idx = np.arange(rows * cols).reshape(rows, cols)
    h = m[:, :-1] & m[:, 1:] & _edges(d[:, :-1], d[:, 1:], diff)
    v = m[:-1, :] & m[1:, :] & _edges(d[:-1, :], d[1:, :], diff)
    src = np.concatenate([idx[:, :-1][h], idx[:-1, :][v]])
    dst = np.concatenate([idx[:, 1:][h], idx[1:, :][v]])
    g = coo_matrix((np.ones(src.size, np.int8), (src, dst)), shape=(rows * cols, rows * cols)).tocsr()
    _, labels = connected_components(g, directed=False)
    mf = m.ravel()
    sizes = np.bincount(labels[mf], minlength=labels.max() + 1)
    speck = mf & (sizes[labels] <= max_speckle_size)
    d.ravel()[speck] = new
    return d, (int(speck.sum()), int(np.unique(labels[speck]).size))


def _opencv_scan(disp, new_value, max_speckle_size, max_diff):
    """Plain-Python port of OpenCV's filterSpecklesImpl (calib3d/src/stereosgbm.cpp) for int16: a row-major scan that
    labels each unlabelled pixel other than newVal with a depth-first wavefront and overwrites small regions as it
    goes. Markers are ordinary values here, as in OpenCV."""
    img = np.array(disp, copy=True)
    new, diff = int(np.rint(new_value)), int(np.rint(max_diff))
    rows, cols = img.shape
    labels = np.zeros((rows, cols), np.int64)
    small = {}
    cur = 0
    for i in range(rows):
        for j in range(cols):
            if img[i, j] == new:
                continue
            if labels[i, j]:
                if small[labels[i, j]]:
                    img[i, j] = new
                continue
            cur += 1
            labels[i, j] = cur
            stack = [(i, j)]
            count = 0
            while stack:
                y, x = stack.pop()
                count += 1
                dp = int(img[y, x])
                for ny, nx in ((y + 1, x), (y - 1, x), (y, x + 1), (y, x - 1)):
                    if 0 <= ny < rows and 0 <= nx < cols and not labels[ny, nx] and img[ny, nx] != new \
                            and abs(dp - int(img[ny, nx])) <= diff:
                        labels[ny, nx] = cur
                        stack.append((ny, nx))
            small[cur] = count <= max_speckle_size
            if small[cur]:
                img[i, j] = new
    return img


# ---------------------------------------------------------------------------------------------- scenes --
def _random_scene(dtype, rows, cols, seed, levels=4, markers=True):
    """Low-entropy values (blobs of every size, many across tile edges), with markers unless told otherwise."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, levels, (rows, cols))
    if np.dtype(dtype) == np.int16:
        d = d.astype(np.int16)
        if markers:
            d[rng.random((rows, cols)) < 0.05] = MARKER
    else:
        d = (d + rng.choice(np.float32([0, 0.25, 0.5]), (rows, cols))).astype(np.float32)
        d[rng.random((rows, cols)) < 0.04] = np.nan
        d[rng.random((rows, cols)) < 0.02] = MARKER
    return d


def _serpentine(dtype, rows, cols):
    """A one-pixel-wide path through the whole frame: every even row, joined at alternate ends."""
    d = np.full((rows, cols), MARKER, dtype)
    d[0::2, :] = 100
    for r in range(1, rows, 2):
        d[r, cols - 1 if (r // 2) % 2 == 0 else 0] = 100
    return d


def _checkerboard(dtype, rows, cols):
    r, c = np.mgrid[0:rows, 0:cols]
    return np.where((r + c) % 2 == 0, 10, 30).astype(dtype)


def _tile_crossers(dtype, rows, cols):
    """On a background of singletons (a checkerboard 1000 / 3000): a 4 x 4 square on every tile corner, a 1 x 6 bar
    across every vertical tile edge and a 6 x 1 bar across every horizontal one, each 16 or 6 pixels of one value."""
    d = np.where((np.add.outer(np.arange(rows), np.arange(cols))) % 2 == 0, 1000, 3000).astype(dtype)
    for y in range(TILE_H, rows, TILE_H):
        for x in range(TILE_W, cols, TILE_W):
            d[y - 2:y + 2, x - 2:x + 2] = 7
    for y in range(4, rows - 1, TILE_H):
        for x in range(TILE_W, cols, TILE_W):
            d[y, x - 3:x + 3] = 9
    for y in range(TILE_H, rows, TILE_H):
        for x in range(40, cols, TILE_W):
            d[y - 3:y + 3, x] = 11
    return d


def _cases():
    """(name, disparity, new_value, max_speckle_size, max_diff) for the restatement checks on the CPU."""
    out = []
    for dtype in (np.int16, np.float32):
        t = np.dtype(dtype).name
        out += [(f"random_{t}", _random_scene(dtype, 23, 41, 1), MARKER, 6, 0),
                (f"random1_{t}", _random_scene(dtype, 20, 37, 2, levels=7), MARKER, 10, 1),
                (f"diff0_{t}", _random_scene(dtype, 17, 19, 3), MARKER, 5, 0),
                (f"diffneg_{t}", _random_scene(dtype, 17, 19, 4), MARKER, 5, -1),
                (f"size0_{t}", _random_scene(dtype, 9, 13, 5), MARKER, 0, 3),
                (f"sizeneg_{t}", _random_scene(dtype, 9, 13, 6), MARKER, -4, 3),
                (f"sizeall_{t}", _random_scene(dtype, 9, 13, 7), MARKER, 9 * 13, 3),
                (f"crossers_{t}", _tile_crossers(dtype, 40, 300), MARKER, 16, 0),
                (f"serpentine_{t}", _serpentine(dtype, 9, 15), MARKER, 68, 0)]
    ext = np.random.default_rng(8).choice(np.int16([32767, -32767, 0, 1, -1]), (15, 21))
    out += [("extremes_65534", ext, MARKER, 5, 65534), ("extremes_65533", ext, MARKER, 5, 65533),
            ("extremes_32767", ext, MARKER, 5, 32767), ("ties_low", _random_scene(np.int16, 15, 21, 9, 6, False), 2.5, 4, 1.5),
            ("ties_high", _random_scene(np.int16, 15, 21, 10, 6, False), 3.5, 4, 0.5),
            ("ties_neg", _random_scene(np.int16, 15, 21, 11, 6), -32768.5, 4, 2.5)]
    return out


# ------------------------------------------------------------------------------------------------ CPU --
@pytest.mark.parametrize("case", [c for c in _cases() if c[1].dtype == np.int16], ids=lambda c: c[0])
def test_restatement_equals_the_opencv_scan(case):
    _, d, new_value, size, diff = case  # OpenCV's filter takes int16 (and uint8) only
    want = _opencv_scan(d, new_value, size, diff)
    got, (pixels, speckles) = _filter(d, new_value, size, diff)
    assert np.array_equal(got, want)
    assert pixels == int((got != d).sum())  # every pixel set was a member, so it differs from `new`
    assert speckles <= pixels


def test_restatement_equals_stored_cv2_outputs():
    z = np.load(GOLDEN)
    names = sorted(k[:-3] for k in z.files if k.endswith("_in"))
    assert len(names) >= 14
    for name in names:
        new_value, size, diff = z[name + "_prm"]
        got, _ = _filter(z[name + "_in"], new_value, int(size), diff)
        assert np.array_equal(got, z[name + "_out"]), name


def test_restatement_equals_live_cv2():
    cv2 = pytest.importorskip("cv2")
    for name, d, new_value, size, diff in _cases():
        if d.dtype != np.int16 or abs(diff) > 32767:  # OpenCV's IPP path truncates maxDiff to int16
            continue
        want, _ = cv2.filterSpeckles(d.copy(), new_value, size, diff)
        assert np.array_equal(_filter(d, new_value, size, diff)[0], want), name
    for seed, shape in enumerate([(480, 640), (1536, 2048)]):
        d = _random_scene(np.int16, *shape, seed=40 + seed, levels=3)
        for size, diff in ((30, 0), (300, 1)):
            want, _ = cv2.filterSpeckles(d.copy(), MARKER, size, diff)
            assert np.array_equal(_filter(d, MARKER, size, diff)[0], want), (shape, size, diff)


def test_scenes_reach_their_edge_cases():
    d = _tile_crossers(np.int16, 40, 300)
    kept, _ = _filter(d, MARKER, 15, 0)
    assert (kept == 7).sum() == 16 * 2 * 2 and (kept == 9).sum() == 0 and (kept == 11).sum() == 0  # only the squares stay
    removed, _ = _filter(d, MARKER, 16, 0)
    assert not np.isin(removed, [7, 9, 11]).any()
    s = _serpentine(np.int16, 9, 15)
    n = int((s == 100).sum())
    assert _filter(s, MARKER, n - 1, 0)[1] == (0, 0) and _filter(s, MARKER, n, 0)[1] == (n, 1)
    c = _checkerboard(np.int16, 6, 7)
    assert _filter(c, MARKER, 1, 19)[1] == (42, 42) and _filter(c, MARKER, 1, 20)[1] == (0, 0)


def test_float_edges_use_the_rounded_difference():
    # exact |a - b| = 1 + 2^-23 + 2^-25 > diff, the float32 difference rounds to 1 + 2^-23 = diff: an edge
    a, b = np.float32(1 + 2.0 ** -23), np.float32(-(2.0 ** -25))
    diff = float(np.float32(1 + 2.0 ** -23))
    assert float(a) - float(b) > diff and np.float32(a - b) == np.float32(diff)
    d = np.array([[a, b]], np.float32)
    assert _filter(d, MARKER, 1, diff)[1] == (0, 0)  # one component of two
    assert _filter(d, MARKER, 2, diff)[1] == (2, 1)
    assert _filter(d, MARKER, 1, np.nextafter(np.float32(diff), np.float32(0)))[1] == (2, 2)
    # overflow to inf: 3e38 - (-3e38) is inf, so only an infinite diff joins them
    big = np.array([[3e38, -3e38]], np.float32)
    assert _filter(big, MARKER, 1, 3.4e38)[1] == (2, 2) and _filter(big, MARKER, 1, np.inf)[1] == (0, 0)
    # inf - inf is NaN: no edge even with an infinite diff; inf - finite is inf
    infs = np.array([[np.inf, np.inf, 5.0, -np.inf]], np.float32)
    assert _filter(infs, MARKER, 1, np.inf)[1] == (1, 1)  # the two +inf apart, 5 joined to its neighbours
    # markers and `new` are never members; NaN new is allowed and matches nothing
    m = np.array([[1, np.nan, MARKER, 7, 1]], np.float32)
    got, c = _filter(m, 7.0, 2, 100)
    assert c == (2, 2) and got[0, 0] == 7 and got[0, 4] == 7 and np.isnan(got[0, 1]) and got[0, 2] == MARKER
    got, c = _filter(m, np.nan, 2, 100)  # 7 is a member now, joined to its neighbour 1
    assert c == (3, 2) and np.isnan(got[0, [0, 1, 3, 4]]).all() and got[0, 2] == MARKER


def test_markers_are_never_members():
    d = np.array([[5, MARKER, MARKER, 5]], np.int16)
    got, c = _filter(d, 0, 2, 0)
    assert c == (2, 2) and list(got[0]) == [0, MARKER, MARKER, 0]  # OpenCV would join and count the markers
    assert list(_opencv_scan(d, 0, 2, 0)[0]) == [0, 0, 0, 0]


def test_speckle_check_binary_is_built():
    assert os.path.exists(CHECK)
    assert "bicos_b200_filter_speckles" in lb.capi.EXPORTS


def test_speckles_take_opencv_types(tmp_path):
    """-DBICOS_WITH_OPENCV: filter_speckles takes a cv::cuda::GpuMat and a cv::cuda::Stream&. Compile-only, against
    the stand-in headers of oracle/shim."""
    src = tmp_path / "speckles_opencv.cpp"
    src.write_text("""#include <BICOS/speckles.hpp>
void calls(cv::cuda::GpuMat& disparity) {
    cv::cuda::Stream stream;
    BICOS::SpeckleCounts n;
    BICOS::filter_speckles(disparity, -32768.0, 100, 1.0);
    BICOS::filter_speckles(disparity, -32768.0, 100, 1.0, &n, stream);
    BICOS::filter_speckles(disparity, 0.0, 100, 1.0, nullptr, static_cast<void*>(nullptr));
    (void)n.pixels;
    (void)n.speckles;
}
""")
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-DBICOS_WITH_OPENCV", "-I" + os.path.join(ROOT, "oracle", "shim"),
           "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include", str(src)]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


# ------------------------------------------------------------------------------------------------ GPU --
def _cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


GUARD = 64


def _run_padded(handle, disp, new_value, size, diff):
    """One call through the C ABI on a padded pitch with guard words before, after and in the padding; returns the
    filtered disparity and the counts, and checks the guards and the launch count."""
    import torch

    rows, cols = disp.shape
    es = disp.dtype.itemsize
    pad = 8 // es + 3
    guard = np.array(-1234, disp.dtype) if disp.dtype == np.int16 else np.float32(-7.25)
    buf = np.full(2 * GUARD + rows * (cols + pad), guard, disp.dtype)
    buf[GUARD:GUARD + rows * (cols + pad)].reshape(rows, cols + pad)[:, :cols] = disp
    d = _cuda(buf)
    counts = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    L = lb.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    before = handle.kernel_launches
    rc = L.bicos_b200_filter_speckles(handle._h, d.data_ptr() + GUARD * es, 3 if disp.dtype == np.int16 else 5,
                                      (cols + pad) * es, rows, cols, float(new_value), int(size), float(diff),
                                      counts.data_ptr(), st)
    assert rc == 0, L.bicos_b200_last_error().decode()
    assert handle.kernel_launches == before + 4
    out = d.cpu().numpy()
    assert (out[:GUARD] == guard).all() and (out[-GUARD:] == guard).all(), "guard words overwritten"
    body = out[GUARD:-GUARD].reshape(rows, cols + pad)
    assert (body[:, cols:] == guard).all(), "pitch padding overwritten"
    return body[:, :cols].copy(), tuple(int(v) for v in counts.cpu())


def _assert_same(got, want):
    g, gc = got
    w, wc = want
    assert gc == wc
    assert g.tobytes() == w.tobytes() or (g.dtype == np.float32 and np.array_equal(g, w, equal_nan=True)
                                          and np.array_equal(np.signbit(g), np.signbit(w)))


SHAPES = [(1, 1), (1, 32767), (32767, 1), (7, 3), (37, 1001), (129, 257), (1536, 2048)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
def test_speckles_bit_exact(handle, shape, dtype):
    rows, cols = shape
    disp = _random_scene(dtype, rows, cols, seed=rows * 3 + cols)
    for size, diff in ((6, 0), (40, 1), (1, 0), (0, 1), (rows * cols, 0), (5, -1)):
        want = _filter(disp, MARKER, size, diff)
        got = _run_padded(handle, disp, MARKER, size, diff)
        try:
            _assert_same(got, want)
        except AssertionError as e:
            raise AssertionError(f"size {size}, diff {diff}: {e}") from None


@pytest.mark.gpu
@pytest.mark.parametrize("case", _cases(), ids=lambda c: c[0])
def test_speckles_bit_exact_constructed(handle, case):
    _, d, new_value, size, diff = case
    _assert_same(_run_padded(handle, d, new_value, size, diff), _filter(d, new_value, size, diff))


@pytest.mark.gpu
def test_speckles_match_stored_cv2_outputs(handle):
    z = np.load(GOLDEN)
    for name in sorted(k[:-3] for k in z.files if k.endswith("_in")):
        new_value, size, diff = z[name + "_prm"]
        got, _ = _run_padded(handle, z[name + "_in"], new_value, int(size), diff)
        assert np.array_equal(got, z[name + "_out"]), name


@pytest.mark.gpu
def test_float_special_values(handle):
    rng = np.random.default_rng(3)
    specials = np.float32([np.nan, MARKER, 7.0, np.inf, -np.inf, 3e38, -3e38, 1 + 2.0 ** -23, -(2.0 ** -25), 0.0, -0.0])
    d = rng.choice(specials, (300, 700)).astype(np.float32)
    d[rng.random(d.shape) < 0.3] = 1.0
    for new_value in (7.0, np.nan, MARKER):
        for diff in (1 + 2.0 ** -23, np.inf, 3.4e38, 0.0):
            _assert_same(_run_padded(handle, d, new_value, 3, diff), _filter(d, new_value, 3, diff))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
@pytest.mark.parametrize("scene", ["serpentine", "covering", "checkerboard", "crossers"])
def test_adversarial_connectivity(handle, dtype, scene):
    rows, cols = 1536, 2048
    d = {"serpentine": _serpentine, "checkerboard": _checkerboard, "crossers": _tile_crossers,
         "covering": lambda t, r, c: np.full((r, c), 42, t)}[scene](dtype, rows, cols)
    n = {"serpentine": int((d == 100).sum()), "covering": rows * cols, "checkerboard": 1, "crossers": 16}[scene]
    for size in (n - 1, n):
        want = _filter(d, MARKER, size, 0)
        _assert_same(_run_padded(handle, d, MARKER, size, 0), want)
        if size == n:
            assert want[1][0] > 0
        elif scene != "crossers":  # the crossers' background singletons go at any size
            assert want[1] == (0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.9, min_variance=2.0),
                                dict(nxcorr_threshold=0.9, subpixel_step=0.1, consistency=True, max_lr_diff=1)])
def test_speckles_of_real_matches(handle, kw):
    left, right, _ = synth.make_stacks(33, 512, 400, np.uint8, seed=3, row0=200, rows=64)
    disp, _ = handle.match(_cuda(left), _cuda(right), Config(**kw))
    host = disp.cpu().numpy()
    new_value = np.nan if "subpixel_step" in kw else MARKER
    for size, diff in ((100, 1), (1000, 1), (20, 0.25)):
        want = _filter(host, new_value, size, diff)
        got = handle.filter_speckles(disp.clone(), new_value, size, diff, counts=True)
        _assert_same((got[0].cpu().numpy(), (got[1]["pixels"], got[1]["speckles"])), want)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
def test_filtering_twice_equals_once(handle, dtype):
    d = _cuda(_random_scene(dtype, 777, 1111, seed=9))
    once = handle.filter_speckles(d, MARKER, 25, 0).clone()
    twice, c = handle.filter_speckles(d, MARKER, 25, 0, counts=True)
    assert c == dict(pixels=0, speckles=0)
    assert np.array_equal(once.cpu().numpy(), twice.cpu().numpy(), equal_nan=True)


@pytest.mark.gpu
def test_errors_launch_nothing(handle):
    import torch

    L = lb.lib()
    d16 = torch.zeros((8, 12), dtype=torch.int16, device="cuda")
    counts = torch.zeros((3,), dtype=torch.int64, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rc(h=None, disp=d16.data_ptr(), typ=3, pitch=24, rows=8, cols=12, new=-32768.0, size=10, diff=1.0,
           c=counts.data_ptr()):
        return L.bicos_b200_filter_speckles(handle._h if h is None else h, disp, typ, pitch, rows, cols, new, size, diff, c, st)

    before = handle.kernel_launches
    bad = [dict(h=ctypes.c_void_p()), dict(disp=None), dict(typ=0), dict(typ=2), dict(typ=6), dict(pitch=22),
           dict(pitch=25), dict(rows=0), dict(cols=0), dict(rows=32768), dict(cols=32768, pitch=65536),
           dict(typ=5, pitch=46), dict(disp=d16.data_ptr() + 1), dict(typ=5, disp=d16.data_ptr() + 2, pitch=48),
           dict(new=32767.5), dict(new=-32769.0), dict(new=float("nan")), dict(new=float("inf")),
           dict(diff=float("nan")), dict(typ=5, pitch=48, diff=float("nan")), dict(c=counts.data_ptr() + 4)]
    for b in bad:
        assert rc(**b) == -1, b
        assert L.bicos_b200_last_error().decode()
    assert handle.kernel_launches == before, "a rejected call launched something"
    assert rc() == 0 and handle.kernel_launches == before + 4
    assert rc(c=None) == 0 and handle.kernel_launches == before + 8
    assert rc(new=32766.5, size=0) == 0 and rc(typ=5, pitch=48, new=float("nan")) == 0  # 32766 fits; NaN for float
    assert handle.kernel_launches == before + 16
    torch.cuda.synchronize()
    with pytest.raises(lb.BicosError, match="int16 or float32"):
        handle.filter_speckles(torch.zeros((4, 4), dtype=torch.float64, device="cuda"), 0, 10, 1)


@pytest.mark.gpu
def test_two_streams_through_one_handle(handle):
    """A call on another stream than the handle's previous call waits for it: the shared labels are not overwritten
    while in use, and both results are complete."""
    import torch

    a0 = _random_scene(np.float32, 1536, 2048, seed=21)
    b0 = _random_scene(np.float32, 1536, 2048, seed=22)
    want_a, want_b = _filter(a0, MARKER, 50, 0), _filter(b0, MARKER, 50, 0)
    a, b = _cuda(a0), _cuda(b0)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        handle.filter_speckles(a, MARKER, 50, 0)
    with torch.cuda.stream(s2):
        handle.filter_speckles(b, MARKER, 50, 0)
    torch.cuda.synchronize()
    assert np.array_equal(a.cpu().numpy(), want_a[0], equal_nan=True)
    assert np.array_equal(b.cpu().numpy(), want_b[0], equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
def test_cpp_filter_speckles(tmp_path, handle, dtype):
    rows, cols = 45, 301
    disp = _random_scene(dtype, rows, cols, seed=31)
    for new_value, size, diff in ((MARKER, 12, 0), (2.5, 30, 1.5)):
        with open(tmp_path / "in.bin", "wb") as f:
            f.write(struct.pack("<4i2d", rows, cols, 3 if disp.dtype == np.int16 else 5, size, new_value, diff))
            f.write(np.ascontiguousarray(disp).tobytes())
        res = subprocess.run([CHECK, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                             timeout=300)
        assert res.returncode == 0, res.stderr
        raw = open(tmp_path / "out.bin", "rb").read()
        counts = struct.unpack("<2Q", raw[:16])
        got = np.frombuffer(raw, disp.dtype, rows * cols, 16).reshape(rows, cols)
        _assert_same((got, counts), _filter(disp, new_value, size, diff))


def _write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]) + img.tobytes())


@pytest.mark.gpu
# SIZE:DIFF per mode, chosen so that each scene has speckles: at DIFF 1 the thresholded disparities of this scene are
# one smooth region each, so the integer mode with a threshold uses DIFF 0 and the subpixel mode a fractional DIFF
@pytest.mark.parametrize("args,new_value,size,diff", [
    (["-t", "0", "-v", "0", "--limited"], MARKER, 30, 1),
    (["-t", "0.9", "-v", "2.0", "--limited"], MARKER, 30, 0),
    (["-t", "0.9", "-v", "2.0", "--limited", "-s", "0.1"], np.nan, 30, 0.25),
])
def test_cli_speckles(tmp_path, handle, args, new_value, size, diff):
    cv2 = pytest.importorskip("cv2")  # reads the CLI's TIFF
    n, rows, cols = 20, 40, 208
    left, right, _ = synth.make_stacks(n, 256, cols, np.uint8, seed=17, row0=100, rows=rows)
    folder = tmp_path / "in"
    folder.mkdir()
    for t in range(n):
        _write_pgm(folder / f"{t}_left.pgm", left[t])
        _write_pgm(folder / f"{t}_right.pgm", right[t])

    def run(extra, out):
        res = subprocess.run([CLI, str(folder), "-o", str(tmp_path / out), *args, *extra], capture_output=True, text=True,
                             timeout=300)
        return res

    plain = run([], "plain.png")
    assert plain.returncode == 0, plain.stderr
    filt = run(["--speckles", f"{size}:{diff}"], "filt.png")
    assert filt.returncode == 0, filt.stderr
    raw = cv2.imread(str(tmp_path / "plain.tiff"), cv2.IMREAD_UNCHANGED)
    got = cv2.imread(str(tmp_path / "filt.tiff"), cv2.IMREAD_UNCHANGED)
    want, (pixels, speckles) = _filter(raw, new_value, size, diff)
    if want.dtype == np.float32:
        want[want == MARKER] = np.nan  # the CLI writes integer-mode markers as NaN
    assert pixels > 0
    assert np.array_equal(got, want, equal_nan=True)
    assert re.search(rf"Removed {speckles} speckles \({pixels} pixels\)", filt.stdout), filt.stdout
    for bad in ("30", "30:", ":1", "x:1", "30:1x", "30:nan", "3.5:1"):
        res = run(["--speckles", bad], "bad.png")
        assert res.returncode != 0 and "speckles" in res.stderr, bad
