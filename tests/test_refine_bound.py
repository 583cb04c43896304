"""The bound that prunes the uint8 refine screen's x steps (refine.cu, the note above refine_kernel; restated in
tools/refine_candidates.py kernel_bound), and the pruned screen on scenes that stress it.

On the CPU: the exact correlation of the kernel's rounded bytes lies below the bound, computed in float32 with its
approximate square roots pushed the wrong way, over random and adversarial stacks; the wrap test flags every pixel
whose rounded values leave [0, 255]; and on bench rows the bound keeps every candidate of the screen.
On the GPU: scenes made of pixels whose parabolas leave [0, 255] (no bound), nearly constant stacks (every step
survives), warps whose lanes keep very different numbers of steps, and the min-variance boundary, bit-identical to the
oracle at 20, 9 and 7 steps (bounded) and at 201 (more than the kernel bounds: every step screened).
"""

import importlib.util
import os

import numpy as np
import pytest

from libbicos_b200 import Config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def _tool():
    spec = importlib.util.spec_from_file_location("refine_candidates", os.path.join(ROOT, "tools", "refine_candidates.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _rounded(y0, y1, y2, x):
    """the kernel's rounded values at step x: ((a x) x + b x) + c in float32, round half even, unwrapped"""
    a = F32(0.5) * (y0 - 2 * y1 + y2).astype(F32)
    b = F32(0.5) * (y2 - y0).astype(F32)
    v = ((a * x) * x + b * x) + y1.astype(F32)
    return np.rint(v).astype(np.int64)


def _stacks(rng, n, p, kind):
    """left and right (columns c1 - 1, c1, c1 + 1) stacks [n, p] of one kind"""
    def u(lo, hi, shape=(n, p)):
        return rng.integers(lo, hi + 1, size=shape)

    if kind == 0:  # random
        y = [u(0, 255) for _ in range(3)]
        li = u(0, 255)
    elif kind == 1:  # dark and bright: parabolas that overshoot, or come close to, either end of the byte range
        lo = rng.random((1, p)) < 0.5
        y = [np.where(lo, u(0, 12), u(243, 255)) for _ in range(3)]
        y[1] = np.where(lo, u(0, 3), u(252, 255))
        li = u(0, 255)
    elif kind == 2:  # left = right interpolated at a random step: correlations near 1 (bytes that cannot wrap)
        y = [u(32, 223) for _ in range(3)]
        x = F32(rng.uniform(-1, 1))
        li = np.clip(_rounded(*y, x) + u(-1, 1) * (rng.random((n, p)) < 0.1), 0, 255)
    elif kind == 3:  # nearly constant right stacks: tiny var_q, s >= 1
        base = u(0, 255, (1, p))
        y = [np.clip(base + u(0, 1) * (rng.random((n, p)) < 0.2), 0, 255) for _ in range(3)]
        li = u(0, 255)
    elif kind == 4:  # constant images, two-valued stacks and their negatives
        base = u(0, 255, (1, p))
        y = [np.broadcast_to(base, (n, p)).copy() for _ in range(3)]
        y[rng.integers(0, 3)][rng.integers(0, n)] ^= 1
        li = 255 - y[1] if rng.random() < 0.5 else y[0].copy()
        li[0] = (li[0] + 1) % 256
    else:  # anticorrelated and correlated with noise
        y = [u(32, 223) for _ in range(3)]
        x = F32(rng.uniform(-1, 1))
        sign = rng.choice([-1, 1])
        li = np.clip(127 + sign * (_rounded(*y, x) - 127) + u(-8, 8), 0, 255)
    return li.astype(np.int64), [v.astype(np.int64) for v in y]


def _exact_rho(li, v):
    n = li.shape[0]
    cov = n * (li * v).sum(0) - li.sum(0) * v.sum(0)
    var0 = n * (li * li).sum(0) - li.sum(0) ** 2
    var1 = n * (v * v).sum(0) - v.sum(0) ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        return cov / np.sqrt(var0.astype(np.float64) * var1)


@pytest.mark.parametrize("n", [9, 17, 33, 65])
def test_exact_score_within_the_bound(n):
    kernel_bound = _tool().kernel_bound
    rng = np.random.default_rng(n)
    # the x values of steps 0.1 and 0.3, both ends, and random floats in [-1, 1]
    fixed = np.concatenate([_tool().steps(0.1), _tool().steps(0.3), np.array([-1, 1], F32)])
    pairs, wrapped, bounded_steps, chunk = 0, 0, 0, 20_000 if n <= 33 else 10_000
    while pairs < 2_000_000:
        kind = (pairs // chunk) % 6
        li, (y0, y1, y2) = _stacks(rng, n, chunk, kind)
        xs = np.concatenate([rng.choice(fixed, 3, replace=False), rng.uniform(-1, 1, 2).astype(F32)])
        wraps, ub, _ = kernel_bound(li, y0, y1, y2, xs)
        for i, x in enumerate(xs):
            v = _rounded(y0, y1, y2, x)
            out = ((v < 0) | (v > 255)).any(0)
            assert not (out & ~wraps).any(), f"n={n} x={x}: a wrapping pixel passed the wrap test"
            rho = _exact_rho(li, v & 0xFF)
            use = ~wraps & np.isfinite(rho)
            bad = use & (rho > ub[i])
            assert not bad.any(), f"n={n} kind={kind} x={x}: rho {rho[bad][0]!r} above its bound {ub[i][bad][0]!r}"
            bounded_steps += int((use & (ub[i] < 2)).sum())
        wrapped += int(wraps.sum())
        pairs += chunk * len(xs)
    assert wrapped > 0, "the dark and bright stacks should wrap sometimes"
    assert bounded_steps > pairs // 5, "the bound should apply to many steps, or the test proves little"


def test_survivors_include_every_candidate_on_bench_rows():
    """tools/refine_candidates.py --bound asserts exact score <= bound for every pixel; the candidates are the steps
    within the margin of the best exact score, so they survive."""
    import json
    import subprocess
    import sys

    for row0 in (100, 1400):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "refine_candidates.py"), "--row0", str(row0),
                              "--rows", "8", "--bound"], check=True, capture_output=True, text=True).stdout
        res = json.loads(out)
        assert res["pixels"] > 10_000
        assert res["survivors_per_pixel"]["mean"] < 4, res
        assert res["rounds_per_warp"]["mean"] < res["rounds_per_warp"]["unpruned"] / 2, res


# ------------------------------------------------------------------------------------------------- GPU scenes --
def _cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _scene(n, rows, cols, seed):
    """Bands of rows: dark and bright right stacks whose parabolas leave [0, 255] (wrap pixels); left equal to the
    right stack, so that correlations near 1 come with narrow bounds; nearly constant right stacks (s >= 1: every
    step survives); and a band whose columns alternate between a smooth and a noisy right stack, so that the lanes of
    a warp keep very different numbers of steps."""
    rng = np.random.default_rng(seed)
    left = rng.integers(0, 256, size=(n, rows, cols)).astype(np.uint8)
    right = rng.integers(0, 256, size=(n, rows, cols)).astype(np.uint8)
    b = rows // 4
    right[:, 0:b] = np.where(rng.random((1, b, cols)) < 0.5, rng.integers(0, 6, (n, b, cols)),
                             rng.integers(250, 256, (n, b, cols))).astype(np.uint8)
    left[:, 0:b] = right[:, 0:b]
    left[:, b:2 * b] = right[:, b:2 * b]
    right[:, 2 * b:3 * b] = (90 + rng.integers(0, 2, size=(n, b, cols))).astype(np.uint8)
    smooth = np.cumsum(rng.integers(-3, 4, size=(n, b, cols)), axis=2) % 256
    band = slice(3 * b, 4 * b)
    right[:, band, ::2] = smooth[:, :, ::2].astype(np.uint8)
    left[:, band] = right[:, band]
    return left, right


def _check(handle, oracles, left, right, kw):
    cfg = Config(**kw)
    disp, corr = handle.match(_cuda(left), _cuda(right), cfg)
    want_d, want_c = oracles.port.match(left, right, **kw)
    got_d, got_c = disp.cpu().numpy(), corr.cpu().numpy()
    evaluated = ~np.isnan(want_c)
    assert evaluated.mean() > 0.3, "the scene should refine most pixels"
    assert np.array_equal(got_c, want_c, equal_nan=True), f"{(got_c != want_c)[evaluated].sum()} corrmap cells differ"
    assert np.array_equal(got_d, want_d, equal_nan=True), f"{(got_d != want_d)[evaluated].sum()} disparities differ"


BASE = dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=4096, no_dupes=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [9, 17, 33, 12, 40, 65])
@pytest.mark.parametrize("step", [0.01, 0.1, 0.25, 0.3])  # 201, 20, 9 and 7 steps
def test_pruned_screen_parity(handle, oracles, n, step):
    left, right = _scene(n, 32, 192, seed=n * 100 + int(step * 100))
    _check(handle, oracles, left, right, dict(BASE, subpixel_step=step))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [9, 33])
def test_pruned_screen_parity_at_min_variance_boundary(handle, oracles, n):
    left, right = _scene(n, 32, 192, seed=5 + n)
    # the nearly constant band's right stacks have var_n near n * p (1 - p) * n for p = 1/2
    for mv in (0.2, 0.25, 0.2499999, 0.2500001):
        _check(handle, oracles, left, right, dict(BASE, subpixel_step=0.1, min_variance=mv))
