"""Reprojection on the device: bicos_b200_reproject, BICOS::reproject / reproject_points, Handle.reproject[_points]
and bicos-cli -q.

The reference is _reproject below, a numpy restatement of the semantics include/bicos_b200.h states (those of
bicos-cli's former host loop). CPU: the restatement against a plain-Python port of that loop, constructed pixels that
an FMA-contracted or reciprocal-multiply evaluation gets wrong (checked with exact rational arithmetic), cv2's
reprojectImageTo3D within a few ULPs, and the OpenCV-types compile check of the header. GPU: the kernel bit-exact
against the restatement over disparity kinds, Q matrices, flags, shapes and pitches, on disparities of real matches,
launch counts and errors, the plain-g++ C++ consumer, and the CLI's .xyz file byte for byte.
"""

import ctypes
import math
import os
import struct
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import libbicos_b200 as lb
from libbicos_b200 import Config, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "libbicos_b200", "bin", "bicos-cli")
CHECK = os.path.join(ROOT, "tests", "cpp", "build", "reproject_check")
MARKER = -32768


def _reproject(disp, Q, allow_negative_z=False):
    """Restatement: disparity [rows, cols] int16 / float32 -> (dense [rows, cols, 3] float32 with NaN where skipped,
    points [N, 3] float32 in row-major order, pixel_index [N] int32, counts (kept, invalid, non-finite, negative Z))."""
    disp = np.asarray(disp)
    q = np.asarray(Q, dtype=np.float64).reshape(4, 4)
    rows, cols = disp.shape
    if disp.dtype == np.int16:
        invalid = disp == MARKER
    else:
        invalid = np.isnan(disp) | (disp == np.float32(MARKER))
    r, c = np.mgrid[0:rows, 0:cols]
    in0, in1, in2 = c.astype(np.float64), r.astype(np.float64), np.where(invalid, 0, disp).astype(np.float64)
    with np.errstate(all="ignore"):
        # numpy rounds every float64 product and sum on its own: no contraction
        o = [((q[k, 0] * in0 + q[k, 1] * in1) + q[k, 2] * in2) + q[k, 3] * 1.0 for k in range(4)]
        xyz = np.stack([(o[k] / o[3]).astype(np.float32) for k in range(3)], axis=-1)
    non_finite = ~invalid & ~np.isfinite(xyz).all(axis=-1)
    negative_z = ~invalid & ~non_finite & (xyz[..., 2] < 0) & (not allow_negative_z)
    kept = ~invalid & ~non_finite & ~negative_z
    dense = np.where(kept[..., None], xyz, np.float32(np.nan)).astype(np.float32)
    index = np.flatnonzero(kept.ravel()).astype(np.int32)
    points = xyz.reshape(-1, 3)[index]
    counts = (int(kept.sum()), int(invalid.sum()), int(non_finite.sum()), int(negative_z.sum()))
    return dense, points, index, counts


def _ieee_div(a, b):
    if b == 0.0:
        if a == 0.0 or math.isnan(a):
            return math.nan
        return math.copysign(math.inf, a) * math.copysign(1.0, b)
    return a / b


def _f32(v):
    with np.errstate(all="ignore"):
        return np.float32(v)


def _scalar_cli(disp, Q, allow_negative_z=False):
    """Plain-Python port of bicos-cli's former host loop (Python floats are doubles, each operation rounded)."""
    q = [float(v) for v in np.asarray(Q, dtype=np.float64).ravel()]
    points, index, counts = [], [], [0, 0, 0, 0]
    rows, cols = disp.shape
    for row in range(rows):
        for col in range(cols):
            v = disp[row, col]
            if disp.dtype == np.int16:
                if v == MARKER:
                    counts[1] += 1
                    continue
            elif math.isnan(v) or v == np.float32(MARKER):
                counts[1] += 1
                continue
            inp = (float(col), float(row), float(v), 1.0)
            o = [q[4 * k] * inp[0] + q[4 * k + 1] * inp[1] + q[4 * k + 2] * inp[2] + q[4 * k + 3] * inp[3] for k in range(4)]
            x, y, z = (_f32(_ieee_div(o[k], o[3])) for k in range(3))
            if not (np.isfinite(x) and np.isfinite(y) and np.isfinite(z)):
                counts[2] += 1
                continue
            if not allow_negative_z and z < 0:
                counts[3] += 1
                continue
            counts[0] += 1
            points.append((x, y, z))
            index.append(row * cols + col)
    return np.array(points, dtype=np.float32).reshape(-1, 3), np.array(index, dtype=np.int32), tuple(counts)


# ---------------------------------------------------------------------------------------------- inputs --
def _stereo_q(cols, rows, f=1400.0, tx=-0.12, dcx=3.5):
    """Shaped like cv2.stereoRectify's Q: [[1, 0, 0, -cx], [0, 1, 0, -cy], [0, 0, 0, f], [0, 0, -1/Tx, (cx - cx')/Tx]]."""
    cx, cy = (cols - 1) / 2.0 + 0.37, (rows - 1) / 2.0 - 0.81
    return np.array([[1, 0, 0, -cx], [0, 1, 0, -cy], [0, 0, 0, f], [0, 0, -1.0 / tx, dcx / tx]], dtype=np.float64)


def _fma_midpoint():
    """(Q, pixel (row, col), d) with X exactly the float32 midpoint m = 1 + 2^-24 when each operation is rounded on
    its own (-> 1.0f), and above m when q2 * d is fused with the running sum -1000 (-> 1.0000001f)."""
    d = float(np.float32(37.3))
    m = 1 + 2.0 ** -24
    q2 = (m + 1000) / d
    for _ in range(200):
        sep = (-1000.0 + q2 * d)
        exact = Fraction(q2) * Fraction(d) - 1000
        if sep == m and exact > Fraction(m):
            break
        q2 = np.nextafter(q2, np.inf if sep < m or exact <= Fraction(m) else -np.inf)
    Q = np.array([[-1000.0, 0, float(q2), 0], [0, 1, 0, 0], [0, 0, 0, 1], [0, 0, 0, 1]])
    return Q, (0, 1), np.float32(d)


def _reciprocal_pair():
    """(Q, d) with RN(o0 / d) and RN(o0 * RN(1 / d)) on opposite sides of the float32 midpoint 1 + 2^-24 (or one on it)."""
    m = Fraction(1) + Fraction(1, 2 ** 24)
    for j in range(1000):
        d = float(np.float32(37.3 + 0.01 * j))
        a = float(m * Fraction(d))
        for _ in range(3):
            a = float(np.nextafter(a, -np.inf))
        for _ in range(7):
            if np.float32(a / d) != np.float32(a * (1.0 / d)):
                Q = np.array([[0, 0, 0, a], [0, 0, 0, 1.0], [0, 0, 0, 2.0], [0, 0, 1.0, 0]])
                return Q, np.float32(d)
            a = float(np.nextafter(a, np.inf))
    raise AssertionError("no reciprocal-multiply counterexample near the midpoint")


def _disparities(kind, rows, cols, seed):
    rng = np.random.default_rng(seed)
    if kind == "int16":
        d = rng.integers(-40, 400, (rows, cols)).astype(np.int16)
        d[rng.random((rows, cols)) < 0.2] = MARKER
        d[rng.random((rows, cols)) < 0.03] = 0
    elif kind == "marker":  # integer mode with a threshold
        d = rng.integers(-40, 400, (rows, cols)).astype(np.float32)
        d[rng.random((rows, cols)) < 0.2] = MARKER
        d[rng.random((rows, cols)) < 0.03] = 0
    else:  # subpixel
        d = rng.uniform(-40, 400, (rows, cols)).astype(np.float32)
        d[rng.random((rows, cols)) < 0.2] = np.nan
        d[rng.random((rows, cols)) < 0.02] = MARKER
        d[rng.random((rows, cols)) < 0.02] = 0
        d[rng.random((rows, cols)) < 0.01] = -0.0
    return d


def _q_matrices(rows, cols, seed):
    rng = np.random.default_rng(seed)
    st = _stereo_q(cols, rows)
    w0 = st.copy()
    w0[3] = 0  # W = 0 everywhere: every point non-finite
    negz = st.copy()
    negz[2, 3] = -1400.0
    big = st.copy()
    big[0] = [1e40, 0, 0, 1e30]  # X beyond the float range unless c is small against W
    tiny = st.copy()
    tiny[0] = [1e-41, 0, 0, 3e-43]  # float subnormals
    tiny[1] = [0, 2.5e-39, 0, 0]
    return {"stereo": st, "random": rng.normal(0, 3, (4, 4)), "w0": w0, "negz": negz, "overflow": big, "subnormal": tiny,
            "midpoint": _fma_midpoint()[0], "reciprocal": _reciprocal_pair()[0]}


# ------------------------------------------------------------------------------------------------ CPU --
@pytest.mark.parametrize("kind", ["int16", "marker", "subpixel"])
@pytest.mark.parametrize("allow", [False, True])
def test_restatement_equals_the_scalar_loop(kind, allow):
    disp = _disparities(kind, 9, 23, seed=5)
    for name, Q in _q_matrices(9, 23, seed=2).items():
        dense, points, index, counts = _reproject(disp, Q, allow)
        want_p, want_i, want_c = _scalar_cli(disp, Q, allow)
        assert counts == want_c, name
        assert sum(counts) == disp.size
        assert np.array_equal(index, want_i), name
        assert points.tobytes() == want_p.tobytes(), name
        kept = np.zeros(disp.size, bool)
        kept[index] = True
        assert np.isnan(dense.reshape(-1, 3)[~kept]).all()
        assert dense.reshape(-1, 3)[kept].tobytes() == points.tobytes()


def test_q_matrices_reach_every_outcome():
    disp = _disparities("subpixel", 20, 40, seed=1)
    seen = {name: _reproject(disp, Q)[3] for name, Q in _q_matrices(20, 40, seed=2).items()}
    assert seen["w0"][0] == 0 and seen["w0"][2] > 0
    assert seen["negz"][3] > 0 and seen["stereo"][3] > 0  # negative disparities give negative W
    assert seen["overflow"][2] > seen["stereo"][2]
    _, pts, _, _ = _reproject(disp, _q_matrices(20, 40, seed=2)["subnormal"])
    sub = np.abs(pts[:, :2][pts[:, :2] != 0])
    assert (sub < np.finfo(np.float32).tiny).any(), "no subnormal coordinate"


def test_fma_contraction_changes_the_constructed_pixel():
    Q, (r, c), d = _fma_midpoint()
    q2 = Fraction(float(Q[0, 2]))
    exact = Fraction(-1000) + q2 * Fraction(float(d))
    separate = -1000.0 + float(Q[0, 2]) * float(d)
    fused = float(exact)  # fma(q2, d, -1000): one rounding of the exact value (Fraction -> float rounds to nearest)
    assert separate == 1 + 2.0 ** -24 and fused > separate
    assert np.float32(separate) == np.float32(1.0) and np.float32(fused) == np.nextafter(np.float32(1), np.float32(2))
    disp = np.zeros((1, 2), np.float32)
    disp[r, c] = d
    dense, _, _, _ = _reproject(disp, Q)
    assert dense[r, c, 0] == np.float32(1.0)
    # the issue's form: q3 = -1000 as the constant term, fused with q2 * d
    q2b = 26.83646167652011
    assert -1000.0 + q2b * float(d) == 1 + 2.0 ** -24
    assert np.float32(float(Fraction(q2b) * Fraction(float(d)) - 1000)) == np.nextafter(np.float32(1), np.float32(2))


def test_reciprocal_division_changes_the_constructed_pixel():
    Q, d = _reciprocal_pair()
    disp = np.full((1, 1), d, np.float32)
    dense, _, _, _ = _reproject(disp, Q)
    a = float(Q[0, 3])
    exact = Fraction(a) / Fraction(float(d))
    assert float(exact) == a / float(d)  # the restatement's division is the correctly rounded one
    assert dense[0, 0, 0] == np.float32(a / float(d)) != np.float32(a * (1.0 / float(d)))


def test_restatement_near_opencv_reproject_image_to_3d():
    cv2 = pytest.importorskip("cv2")
    disp = _disparities("subpixel", 48, 64, seed=3)
    disp[disp <= 1] = np.nan  # positive disparities: cv2 and the restatement both keep them
    Q = _stereo_q(64, 48)
    dense, _, _, _ = _reproject(disp, Q)
    cv = cv2.reprojectImageTo3D(np.nan_to_num(disp, nan=-1.0), Q, handleMissingValues=False)
    ok = np.isfinite(dense).all(axis=-1)
    assert ok.sum() > 1000
    ulps = np.abs(dense[ok].view(np.int32).astype(np.int64) - cv[ok].astype(np.float32).view(np.int32).astype(np.int64))
    assert ulps.max() <= 4


def test_reproject_check_binary_is_built():
    assert os.path.exists(CHECK)
    assert "bicos_b200_reproject" in lb.capi.EXPORTS


def test_reproject_takes_opencv_types(tmp_path):
    """-DBICOS_WITH_OPENCV: reproject / reproject_points take cv::cuda::GpuMat and a cv::cuda::Stream&. Compile-only,
    against the stand-in headers of oracle/shim."""
    src = tmp_path / "reproject_opencv.cpp"
    src.write_text("""#include <BICOS/reproject.hpp>
void calls(const cv::cuda::GpuMat& disparity, const std::array<double, 16>& Q) {
    cv::cuda::GpuMat xyz, points, index;
    cv::cuda::Stream stream;
    BICOS::reproject(disparity, Q, xyz);
    BICOS::reproject(disparity, Q, xyz, true, stream);
    BICOS::reproject(disparity, Q, xyz, false, static_cast<void*>(nullptr));
    BICOS::ReprojectCounts n = BICOS::reproject_points(disparity, Q, points);
    n = BICOS::reproject_points(disparity, Q, points, &index, true, stream);
    n = BICOS::reproject_points(disparity, Q, points, nullptr, false, static_cast<void*>(nullptr));
    (void)n.points;
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


SHAPES = [(1, 1), (1, 1025), (7, 3), (37, 1001), (1536, 2048), (1, 32767)]
GUARD = 64


def _run_padded(handle, disp, Q, allow):
    """Dense and point list of one call through the C ABI, with padded disparity and xyz pitches and guard words
    around xyz and beyond the points written; returns (dense, points, index, counts) and checks the guards."""
    import torch

    rows, cols = disp.shape
    es = disp.dtype.itemsize
    pad = 8 // es + 3  # padded pitch, still a multiple of the element size
    dbuf = np.zeros((rows, cols + pad), disp.dtype)
    dbuf[:, :cols] = disp
    d = _cuda(dbuf)
    mark = np.float32(-7.25)
    xyz_pitch = 3 * cols + 5  # floats
    flat = torch.full((GUARD + rows * xyz_pitch + GUARD,), float(mark), dtype=torch.float32, device="cuda")
    pts = torch.full((rows * cols * 3 + GUARD,), float(mark), dtype=torch.float32, device="cuda")
    idx = torch.full((rows * cols + GUARD,), -5, dtype=torch.int32, device="cuda")
    counts = torch.full((4,), -1, dtype=torch.int64, device="cuda")
    L = lb.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    before = handle.kernel_launches
    rc = L.bicos_b200_reproject(handle._h, d.data_ptr(), 3 if disp.dtype == np.int16 else 5, (cols + pad) * es, rows, cols,
                                handle._q_matrix(Q), int(allow), flat.data_ptr() + GUARD * 4, xyz_pitch * 4, pts.data_ptr(),
                                idx.data_ptr(), counts.data_ptr(), st)
    assert rc == 0, L.bicos_b200_last_error().decode()
    assert handle.kernel_launches == before + 1, "dense + points should be one launch"
    f = flat.cpu().numpy()
    assert (f[:GUARD] == mark).all() and (f[-GUARD:] == mark).all(), "guard words around xyz overwritten"
    body = f[GUARD:-GUARD].reshape(rows, xyz_pitch)
    assert (body[:, 3 * cols:] == mark).all(), "xyz pitch padding overwritten"
    c = tuple(int(v) for v in counts.cpu())
    p = pts.cpu().numpy()
    i = idx.cpu().numpy()
    assert (p[3 * c[0]:] == mark).all() and (i[c[0]:] == -5).all(), "points or indices written beyond counts[0]"
    return body[:, : 3 * cols].reshape(rows, cols, 3), p[: 3 * c[0]].reshape(-1, 3), i[: c[0]], c


def _assert_same(got, want):
    gd, gp, gi, gc = got
    wd, wp, wi, wc = want
    assert gc == wc
    assert np.array_equal(np.isnan(gd), np.isnan(wd))
    ok = ~np.isnan(wd)
    assert gd[ok].tobytes() == wd[ok].tobytes()  # bitwise: -0.0 and subnormals included
    assert np.array_equal(gi, wi)
    assert gp.tobytes() == wp.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind", ["int16", "marker", "subpixel"])
def test_reproject_bit_exact(handle, shape, kind):
    rows, cols = shape
    disp = _disparities(kind, rows, cols, seed=rows * 7 + cols)
    Qs = _q_matrices(rows, cols, seed=cols)
    if cols >= 2 and kind != "int16":
        disp[0, 1] = _fma_midpoint()[2]  # the constructed pixels
        disp[0, 0] = _reciprocal_pair()[1]
    for name, Q in Qs.items():
        if rows * cols > 10 ** 6 and name not in ("stereo", "random", "negz", "midpoint"):
            continue  # the big frame: the common shapes; the special matrices run on the others
        for allow in (False, True):
            want = _reproject(disp, Q, allow)
            got = _run_padded(handle, disp, Q, allow)
            try:
                _assert_same(got, want)
            except AssertionError as e:
                raise AssertionError(f"{name}, allow_negative_z={allow}: {e}") from None
            if name == "midpoint" and cols >= 2 and kind != "int16":
                assert got[0][0, 1, 0] == np.float32(1.0), "the constructed pixel was evaluated with a fused multiply-add"


@pytest.mark.gpu
def test_handle_api_and_repeated_calls(handle):
    import torch

    disp = _disparities("subpixel", 1536, 2048, seed=11)
    Q = _stereo_q(2048, 1536)
    want = _reproject(disp, Q)
    d = _cuda(disp)
    dense = handle.reproject(d, Q)
    out = torch.zeros_like(dense)
    assert handle.reproject(d, Q, out=out).data_ptr() == out.data_ptr()
    first = handle.reproject_points(d, torch.tensor(Q))  # Q from a tensor
    for _ in range(3):
        pts, idx, counts = handle.reproject_points(d, Q.tolist())  # and from nested lists
        assert torch.equal(pts, first[0]) and torch.equal(idx, first[1]) and counts == first[2]
    got = (dense.cpu().numpy(), pts.cpu().numpy(), idx.cpu().numpy(),
           (counts["points"], counts["invalid_disparity"], counts["non_finite"], counts["negative_z"]))
    _assert_same(got, want)
    assert np.array_equal(out.cpu().numpy(), dense.cpu().numpy(), equal_nan=True)
    pts_neg, _, c_neg = handle.reproject_points(d, Q, allow_negative_z=True)
    assert c_neg["negative_z"] == 0 and c_neg["points"] == counts["points"] + counts["negative_z"]


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.9, min_variance=2.0),
                                dict(nxcorr_threshold=0.9, subpixel_step=0.1, consistency=True, max_lr_diff=1)])
def test_reproject_of_real_matches(handle, kw):
    left, right, _ = synth.make_stacks(33, 512, 400, np.uint8, seed=3, row0=200, rows=64)
    disp, _ = handle.match(_cuda(left), _cuda(right), Config(**kw))
    host = disp.cpu().numpy()
    assert host.dtype == (np.int16 if kw["nxcorr_threshold"] is None else np.float32)
    Q = _stereo_q(400, 64)
    for allow in (False, True):
        want = _reproject(host, Q, allow)
        assert want[3][0] > 1000
        dense = handle.reproject(disp, Q, allow_negative_z=allow).cpu().numpy()
        pts, idx, c = handle.reproject_points(disp, Q, allow_negative_z=allow)
        _assert_same((dense, pts.cpu().numpy(), idx.cpu().numpy(), tuple(c.values())), want)


@pytest.mark.gpu
def test_reproject_of_match_rectified(handle):
    from libbicos_b200 import RectifyMaps

    left, right, _ = synth.make_stacks(33, 512, 330, np.uint8, seed=4, rows=60)
    maps = []
    for cam in (0, 1):
        mx, my = synth.rectify_maps(48, 320, 60, 330, camera=cam, k1=-0.05, k2=0.0, angle_deg=0.1)
        maps += [_cuda(mx), _cuda(my)]
    disp, _ = handle.match_rectified(_cuda(left), _cuda(right), RectifyMaps(*maps),
                                     Config(nxcorr_threshold=0.9, subpixel_step=0.1, min_variance=2.0))
    Q = _stereo_q(320, 48)
    want = _reproject(disp.cpu().numpy(), Q)
    pts, idx, c = handle.reproject_points(disp, Q)
    _assert_same((handle.reproject(disp, Q).cpu().numpy(), pts.cpu().numpy(), idx.cpu().numpy(), tuple(c.values())), want)


@pytest.mark.gpu
def test_reproject_errors_launch_nothing(handle):
    import torch

    L = lb.lib()
    d16 = torch.zeros((8, 12), dtype=torch.int16, device="cuda")
    xyz = torch.empty((8, 12, 3), dtype=torch.float32, device="cuda")
    pts = torch.empty((96, 3), dtype=torch.float32, device="cuda")
    idx = torch.empty((96,), dtype=torch.int32, device="cuda")
    counts = torch.empty((4,), dtype=torch.int64, device="cuda")
    q = handle._q_matrix(np.eye(4))
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def rc(h=None, disp=d16.data_ptr(), typ=3, pitch=24, rows=8, cols=12, q_=q, flags=0, x=xyz.data_ptr(), xp=144,
           p=pts.data_ptr(), i=idx.data_ptr(), c=counts.data_ptr()):
        return L.bicos_b200_reproject(handle._h if h is None else h, disp, typ, pitch, rows, cols, q_, flags, x, xp, p, i, c, st)

    before = handle.kernel_launches
    bad = [dict(h=ctypes.c_void_p()), dict(q_=None), dict(disp=None), dict(typ=0), dict(typ=2), dict(typ=6), dict(flags=2),
           dict(x=None, p=None, i=None), dict(c=None), dict(p=None), dict(pitch=22), dict(pitch=25), dict(xp=140),
           dict(xp=146), dict(rows=0), dict(cols=0), dict(rows=32768, pitch=24), dict(cols=32768, pitch=65536, xp=32768 * 12),
           dict(typ=5, pitch=46)]
    for b in bad:
        assert rc(**b) == -1, b
        assert L.bicos_b200_last_error().decode()
    assert handle.kernel_launches == before, "a rejected call launched something"
    assert rc() == 0 and handle.kernel_launches == before + 1
    assert rc(p=None, i=None, c=None) == 0 and handle.kernel_launches == before + 2  # dense alone
    assert rc(x=None) == 0 and handle.kernel_launches == before + 3  # list alone
    torch.cuda.synchronize()
    with pytest.raises(lb.BicosError, match="int16 or float32"):
        handle.reproject(torch.zeros((4, 4), dtype=torch.float64, device="cuda"), np.eye(4))
    with pytest.raises(lb.BicosError, match="4 x 4"):
        handle.reproject(d16, np.eye(3))


@pytest.mark.gpu
def test_reproject_follows_the_previous_stream(handle):
    """A call on another stream than the handle's previous call waits for it: the two point lists are complete."""
    import torch

    disp = _cuda(_disparities("subpixel", 1536, 2048, seed=12))
    Q = _stereo_q(2048, 1536)
    want = handle.reproject_points(disp, Q)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        a = handle.reproject_points(disp, Q)
    with torch.cuda.stream(s2):
        b = handle.reproject_points(disp, Q)
    torch.cuda.synchronize()
    for got in (a, b):
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]) and got[2] == want[2]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["int16", "marker", "subpixel"])
def test_cpp_reproject(tmp_path, handle, kind):
    rows, cols = 45, 301
    disp = _disparities(kind, rows, cols, seed=9)
    for allow in (False, True):
        Q = _stereo_q(cols, rows)
        with open(tmp_path / "in.bin", "wb") as f:
            f.write(struct.pack("<4i", rows, cols, 3 if disp.dtype == np.int16 else 5, int(allow)))
            f.write(Q.astype("<f8").tobytes())
            f.write(np.ascontiguousarray(disp).tobytes())
        res = subprocess.run([CHECK, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                             timeout=300)
        assert res.returncode == 0, res.stderr
        raw = open(tmp_path / "out.bin", "rb").read()
        counts = struct.unpack("<4Q", raw[:32])
        n = counts[0]
        dense = np.frombuffer(raw, np.float32, rows * cols * 3, 32).reshape(rows, cols, 3)
        off = 32 + dense.nbytes
        pts = np.frombuffer(raw, np.float32, 3 * n, off).reshape(-1, 3)
        idx = np.frombuffer(raw, np.int32, n, off + pts.nbytes)
        _assert_same((dense, pts, idx, counts), _reproject(disp, Q, allow))


def _write_pgm(path, img):
    hi = 65535 if img.dtype == np.uint16 else 255
    data = img.astype(">u2").tobytes() if img.dtype == np.uint16 else img.tobytes()
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n%d\n" % (img.shape[1], img.shape[0], hi) + data)


@pytest.mark.gpu
@pytest.mark.parametrize("args,kw", [
    (["-t", "0", "-v", "0", "--limited"], dict(nxcorr_threshold=None)),
    (["-t", "0.9", "-v", "2.0", "--limited"], dict(nxcorr_threshold=0.9, min_variance=2.0)),
    (["-t", "0.9", "-v", "2.0", "--limited", "-s", "0.1"], dict(nxcorr_threshold=0.9, min_variance=2.0, subpixel_step=0.1)),
])
@pytest.mark.parametrize("allow", [False, True])
def test_cli_pointcloud_bytes(tmp_path, handle, args, kw, allow):
    n, rows, cols = 20, 40, 208
    left, right, _ = synth.make_stacks(n, 256, cols, np.uint8, seed=17, row0=100, rows=rows)
    folder = tmp_path / "in"
    folder.mkdir()
    for t in range(n):
        _write_pgm(folder / f"{t}_left.pgm", left[t])
        _write_pgm(folder / f"{t}_right.pgm", right[t])
    # W = d - 40: disparities below 40 give negative Z, exactly 40 gives W = 0; X = 1e38 (c - 103.5) / W leaves the
    # float range wherever |c - 103.5| > 3.4 |W|: non-finite points in every disparity kind
    Q = np.array([[1e38, 0, 0, -1.035e40], [0, 1, 0, -19.5], [0, 0, 0, 900.0], [0, 0, 1.0, -40.0]])
    q = tmp_path / "q.yaml"
    q.write_text("%YAML:1.0\n---\nQ: !!opencv-matrix\n   rows: 4\n   cols: 4\n   dt: d\n   data: [ "
                 + ", ".join(repr(float(v)) for v in Q.ravel()) + " ]\n")
    extra = ["--allow-negative-z"] if allow else []
    res = subprocess.run([CLI, str(folder), "-o", str(tmp_path / "d.png"), *args, "-q", str(q), *extra], capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    disp, _ = handle.match(_cuda(left), _cuda(right), Config(**kw))
    _, pts, _, counts = _reproject(disp.cpu().numpy(), Q, allow)
    assert counts[0] > 500 and counts[2] > 0 and (allow or counts[3] > 0)
    want = "".join("%g %g %g\n" % (float(x), float(y), float(z)) for x, y, z in pts)
    assert (tmp_path / "d.xyz").read_bytes() == want.encode()
    lines = [ln for ln in res.stderr.splitlines() if ln.startswith("Skipped")]
    expect = []
    if counts[2]:
        expect.append(f"Skipped {counts[2]} points with non-finite fp values")
    if counts[3]:
        expect.append(f"Skipped {counts[3]} points with negative Z values")
    assert lines == expect
