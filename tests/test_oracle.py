"""CPU tests of the checkers: the C restatement against the golden vectors generated from the
unmodified reference (tests/golden/make_golden.py), against the reference build itself when it
is present, plus the arithmetic facts the CUDA kernels rely on."""

import glob
import os
import zlib

import numpy as np
import pytest

from libbicos_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _cases():
    import importlib.util

    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLDEN, "make_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True) if a.dtype.kind == "f" else np.array_equal(a, b)


def test_golden_files_present():
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
    assert names == sorted(_cases().CASES)


@pytest.mark.parametrize("name", sorted(_cases().CASES))
def test_port_matches_golden(oracles, name):
    mg = _cases()
    case = mg.CASES[name]
    kw = case[7]
    left, right = mg.inputs(case)
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    assert int(g["input_crc"]) == mg.crc(left, right), "synthetic generator changed: regenerate the fixtures"
    full = bool(kw.get("mode_full", False))
    wide = bool(kw.get("wide_descriptors", False))
    d0 = oracles.port.descriptors(left, full, wide)
    d1 = oracles.port.descriptors(right, full, wide)
    assert np.array_equal(d0, g["desc0"]) and np.array_equal(d1, g["desc1"])
    flags = (2 | (1 if kw.get("no_dupes") else 0)) if kw.get("consistency") else 1
    raw = oracles.port.bicos(d0, d1, flags, kw.get("max_lr_diff", 1) if kw.get("consistency") else -1)
    assert np.array_equal(raw, g["raw"])
    disp, corr = oracles.port.match(left, right, **kw)
    assert _same(disp, g["disp"])
    if corr is not None:
        assert _same(corr, g["corr"])
    if kw.get("nxcorr_threshold") is not None:
        # stage-level refine entry point from the golden raw disparity
        d2, c2 = oracles.port.agree(g["raw"], left, right, kw["nxcorr_threshold"], kw.get("subpixel_step"),
                                    kw.get("min_variance"))
        want = g["disp"] if kw.get("subpixel_step") is not None else g["disp"].astype(np.int16)
        assert _same(d2, want) and _same(c2, g["corr"])


def _reference_outputs():
    import importlib.util

    spec = importlib.util.spec_from_file_location("make_reference_outputs", os.path.join(GOLDEN, "make_reference_outputs.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


RO = _reference_outputs()


@pytest.mark.parametrize("n,dtype,full", RO.BUILD_CASES)
def test_port_matches_reference_build(oracles, n, dtype, full):
    """The port against the reference build, or without it against the reference's outputs stored in
    tests/golden/reference/ (tests/golden/make_reference_outputs.py)."""
    live = oracles.ref.available()
    key = f"port_build/{n}_{np.dtype(dtype).name}_{int(full)}"
    left, right = RO.build_inputs(n, dtype)
    desc = oracles.port.descriptors(left, full)
    if live:
        assert np.array_equal(oracles.ref.descriptors(left, full), desc)
    else:
        RO.check_inputs(key, left, right)
        RO.check(f"{key}/desc", desc)
    for i, kw in enumerate(RO.BUILD_KWS):
        b = oracles.port.match(left, right, mode_full=full, **kw)
        if live:
            a = oracles.ref.match(left, right, mode_full=full, **kw)
            assert _same(a[0], b[0])
            assert (a[1] is None and b[1] is None) or _same(a[1], b[1])
        else:
            RO.check(f"{key}/{i}/disp", b[0])
            RO.check(f"{key}/{i}/corr", b[1])


@pytest.mark.parametrize("n,dtype", RO.WIDE_CASES)
def test_wide_extension_matches_reference_stage_templates(oracles, n, dtype):
    """FULL stacks of 17..23 images need 258..486 bits; the reference's driver throws above 256. The port's
    12- and 16-word paths are pinned against the reference's own stage templates with std::bitset<384/512>
    (without the reference build: against their outputs stored in tests/golden/reference/)."""
    live = oracles.ref.available()
    key = f"wide/{n}_{np.dtype(dtype).name}"
    left, right = RO.build_inputs(n, dtype, rows=16)
    k = oracles.words_per_descriptor(n, True, wide=True)
    assert k == (12 if n <= 20 else 16)
    b = oracles.port.descriptors(left, True, wide=True)
    assert b.shape[2] == k
    if live:
        assert np.array_equal(oracles.ref.descriptors(left, True, wide=True), b)
    else:
        RO.check_inputs(key, left, right)
        RO.check(f"{key}/desc", b)
    assert (b[..., 8:] != 0).any(), "the words beyond 256 bits must be in use"
    for i, kw in enumerate(RO.WIDE_KWS):
        y = oracles.port.match(left, right, mode_full=True, wide_descriptors=True, **kw)
        if live:
            x = oracles.ref.match(left, right, mode_full=True, wide_descriptors=True, **kw)
            assert _same(x[0], y[0])
            assert (x[1] is None and y[1] is None) or _same(x[1], y[1])
        else:
            RO.check(f"{key}/{i}/disp", y[0])
            RO.check(f"{key}/{i}/corr", y[1])
    with pytest.raises(RuntimeError, match="too large"):
        oracles.port.match(left, right, mode_full=True)


def test_search_ties_against_reference_build(oracles):
    """Random low-entropy descriptors: many exact ties, all three flag combinations, K = 1..16, against the
    reference build or without it against its results stored in tests/golden/reference/."""
    for k, (d0, d1) in RO.tie_descriptors().items():
        for flags in (1, 2, 3):
            got = oracles.port.bicos(d0, d1, flags, 2)
            want = oracles.ref.bicos(d0, d1, flags, 2) if oracles.ref.available() else RO.stored()[1][f"ties_k{k}_f{flags}"]
            assert np.array_equal(want, got), (k, flags)


def test_errors_follow_reference(oracles):
    one = np.zeros((1, 4, 4), np.uint8)
    with pytest.raises(RuntimeError, match="at least two"):
        oracles.port.match(one, one)
    big = np.zeros((20, 4, 4), np.uint8)
    with pytest.raises(RuntimeError, match="363 bits"):
        oracles.port.match(big, big, mode_full=True)
    if oracles.ref.available():
        with pytest.raises(RuntimeError, match="at least two"):
            oracles.ref.match(one, one)
        with pytest.raises(RuntimeError, match="363 bits"):
            oracles.ref.match(big, big, mode_full=True)


def test_double_path_close_to_float(oracles):
    """The f64 restatement (unpinned arithmetic core) stays within float rounding of the pinned f32 path."""
    left, right, _ = synth.make_stacks(33, 512, 160, np.uint8, seed=8, row0=64, rows=24)
    kw = dict(nxcorr_threshold=0.9, min_variance=2.0)
    df, cf = oracles.port.match(left, right, **kw)
    dd, cd = oracles.port.match(left, right, double=True, **kw)
    assert cd.dtype == np.float64
    ok = ~np.isnan(cf)
    assert np.array_equal(np.isnan(cd), np.isnan(cf))
    assert np.max(np.abs(cd[ok] - cf[ok])) < 1e-5
    assert (dd != df).mean() < 0.01


# ------------------------------------------------------------------ facts the kernels use --
def test_integer_mean_comparison_is_exact():
    """(float)p < fl(sum/n)  <=>  p*n < sum  <=>  p < ceil(sum/n), for n <= 65 and 16-bit pixels."""
    rng = np.random.default_rng(1)
    for n in (2, 3, 5, 9, 17, 33, 34, 64, 65):
        for hi in (256, 65536):
            pix = rng.integers(0, hi, size=(20000, n), dtype=np.int64)
            # near-constant stacks are the hard cases: the mean sits next to the pixel values
            base = rng.integers(0, hi - 2, size=(20000, 1))
            pix[:10000] = base[:10000] + rng.integers(0, 2, size=(10000, n))
            s = pix.sum(axis=1, keepdims=True)
            av = (s.astype(np.float32) / np.float32(n)).astype(np.float32)
            ref = pix.astype(np.float32) < av
            assert np.array_equal(ref, pix * n < s)
            thr = (s + n - 1) // n
            assert np.array_equal(ref, pix < thr)
            m = ((1 << 24) + n - 1) // n
            if hi == 256:
                assert np.array_equal(((s + n - 1) * m) >> 24, thr)  # reciprocal multiply used on the GPU


def test_subpixel_x_sequence():
    """The float loop x=-1; x<=1; x+=0.1f has 20 values, never hits 0 or 1 (SURVEY.md 9.4)."""
    xs = []
    x = np.float32(-1.0)
    step = np.float32(0.1)
    while x <= np.float32(1.0):
        xs.append(x)
        x = np.float32(x + step)
    assert len(xs) == 20 and float(xs[-1]) == pytest.approx(0.900000155, abs=1e-8)
    assert min(abs(float(v)) for v in xs) == pytest.approx(7.45e-8, rel=0.01)


def test_magic_rounding_equals_roundeven_and_wrap():
    """fl(v + 1.5*2^23) rounds half-to-even and leaves the integer in the low mantissa bits."""
    rng = np.random.default_rng(2)
    v = np.concatenate([rng.uniform(-300000, 300000, 200000), np.arange(-2000, 2000) + 0.5,
                        np.arange(-2000, 2000) - 0.5]).astype(np.float32)
    m = (v + np.float32(12582912.0)).astype(np.float32)
    bits = m.view(np.uint32)
    want = np.rint(v.astype(np.float64)).astype(np.int64)  # rint = half to even
    assert np.array_equal((bits & 0xFF).astype(np.int64), want & 0xFF)
    assert np.array_equal((bits & 0xFFFF).astype(np.int64), want & 0xFFFF)
    back = ((bits & 0xFFFF) | np.uint32(0x4B000000)).view(np.float32) - np.float32(8388608.0)
    assert np.array_equal(back.astype(np.int64), want & 0xFFFF)


def test_synth_is_shardable_and_backend_independent():
    import torch

    full = synth.make_stacks(5, 64, 48, np.uint8, seed=3)
    part = synth.make_stacks(5, 64, 48, np.uint8, seed=3, row0=20, rows=11)
    for a, b in zip(full, part):
        assert np.array_equal(a[..., 20:31, :], b)
    for dt in (np.uint8, np.uint16):
        a = synth.make_stacks(4, 40, 33, dt, seed=9, frame=2)
        b = synth.make_stacks(4, 40, 33, dt, seed=9, frame=2, xp=torch, device="cpu")
        assert np.array_equal(a[0], b[0].view(torch.int16).numpy().view(np.uint16) if dt == np.uint16 else b[0].numpy())
        assert np.array_equal(a[2], b[2].numpy())
    assert zlib.crc32(full[0].tobytes()) != zlib.crc32(synth.make_stacks(5, 64, 48, np.uint8, seed=3, frame=1)[0].tobytes())


def test_mean_by_reciprocal_is_the_ieee_quotient():
    """refine.cu computes the float means sum / n as q0 = RN(s r), rem = s - q0 n (one FMA, exact), q = RN(q0 + rem r)
    with r = RN(1 / n) (mean_of_sum) instead of an IEEE division (reference include/impl/cpu/agree.hpp:34-36, cv::mean
    in float): the same float for EVERY integer sum in [0, 65535 n] and every stack size 2 <= n <= 65. Emulated in
    float64, where every intermediate is exact except the last sum; results whose float64 value lies within one
    float64 ulp of a float32 rounding midpoint (where that emulation could round twice) are re-checked in rationals."""
    from fractions import Fraction

    f32 = np.float32
    flagged = 0
    for n in range(2, 66):
        a = np.arange(0, n * 65535 + 1, dtype=np.float64)
        r = np.float64(f32(1.0) / f32(n))
        want = (a.astype(f32) / f32(n)).astype(np.float64)
        q0 = (a * r).astype(f32).astype(np.float64)  # 24 x 24 bits: exact in float64, then RN to float32
        rem = (a - q0 * n).astype(f32).astype(np.float64)  # the FMA's exact value (q0 n: 31 bits; the difference is small)
        t = q0 + rem * r  # rem r exact (48 bits); the sum may round in float64
        assert np.array_equal(t.astype(f32).astype(np.float64), want), n
        low = t.view(np.int64) & ((1 << 29) - 1)  # float64 mantissa bits below float32 precision
        for i in np.nonzero(np.abs(low - (1 << 28)) <= 1)[0]:
            flagged += 1
            exact = Fraction(float(q0[i])) + Fraction(float(rem[i])) * Fraction(float(r))
            lo, hi = f32(np.nextafter(f32(want[i]), f32(-np.inf))), f32(np.nextafter(f32(want[i]), f32(np.inf)))
            assert abs(exact - Fraction(float(want[i]))) <= min(abs(exact - Fraction(float(lo))), abs(exact - Fraction(float(hi))))
    assert flagged == 0  # none today; the branch above stays for other float environments
