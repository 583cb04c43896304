"""The screen of the uint8 float subpixel refine (refine.cu, the note above refine_kernel).

On the CPU: the error bound delta(n) = (2n + 8) 2^-24 of the reference's float NXC chain against the exact correlation,
and the variance margin (n + 5) 2^-24, against the float chain itself on random and adversarial stacks.
On the GPU: scenes made of near ties, small and constant variances and min-variance boundaries, bit-identical to the
oracle.
"""

import ctypes
import os
import subprocess

import numpy as np
import pytest

from libbicos_b200 import Config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24
KINDS = 6  # tools/refine_screen.c draw(): random, nearly constant, minimal variance, anti-, correlated, ties


def _helper():
    path = os.path.join(ROOT, "tools", "librefine_screen.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tools"), path], check=True)
    lib = ctypes.CDLL(path)
    f = lib.rs_worst_error
    f.restype = ctypes.c_long
    f.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_uint64, ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                  ctypes.POINTER(ctypes.c_double)]
    return f


@pytest.mark.parametrize("n", [2, 9, 17, 33, 64, 65])
def test_float_chain_within_half_the_screen_bound(n):
    f = _helper()
    per_kind = 10_000_000 // KINDS + 1
    worst, worst_var, used = 0.0, 0.0, 0
    for kind in range(KINDS):
        e, ev = ctypes.c_double(), ctypes.c_double()
        used += f(n, per_kind, 1000 * n + kind, kind, ctypes.byref(e), ctypes.byref(ev))
        worst, worst_var = max(worst, e.value), max(worst_var, ev.value)
    assert used >= 8_000_000  # stacks with a zero variance (often among the nearly constant ones at n = 2) are left out
    delta, var_margin = 2 * n + 8, n + 5  # in units of 2^-24, refine.cu screen_margin() / var_margin()
    assert worst <= delta / 2, f"n={n}: float NXC off by {worst} u, delta = {delta} u"
    # the kernel tests var1_n against n * minvar * (1 -+ 2 var_margin)
    assert worst_var <= var_margin, f"n={n}: float variance off by {worst_var} u, margin = {var_margin} u"


# ------------------------------------------------------------------------------------------------- GPU scenes --
def _cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _scene(n, rows, cols, seed):
    """Bands of rows, each a structure of the right stack around the matched columns (the left stack is random):
    symmetric neighbourhoods (steps x and -x tie), nearly constant and constant stacks, two-valued stacks with the
    smallest nonzero variance (the min-variance boundary), and stacks constant along the row, where every step has
    the same values (more than two candidates: the unscreened loop)."""
    rng = np.random.default_rng(seed)
    left = rng.integers(0, 256, size=(n, rows, cols)).astype(np.uint8)
    right = rng.integers(0, 256, size=(n, rows, cols)).astype(np.uint8)
    b = rows // 5
    # 0: every even column equals column 0 (per image and row): y(c1 - 1) == y(c1 + 1) at odd c1
    right[:, 0:b, 2::2] = right[:, 0:b, 0:1]
    # 1: nearly constant, constant in some columns
    right[:, b:2 * b] = (100 + rng.integers(0, 2, size=(n, b, cols))).astype(np.uint8)
    right[:, b:2 * b, ::7] = 100
    # 2: two values, one of them in one image only: var_n = n - 1
    right[:, 2 * b:3 * b] = 37
    right[rng.integers(0, n, size=(b, cols)), np.arange(2 * b, 3 * b)[:, None], np.arange(cols)[None, :]] = 38
    # 3: constant along the row
    right[:, 3 * b:4 * b] = right[:, 3 * b:4 * b, 0:1]
    # 4: random; left equal to right, so that correlations near 1 and their ties occur
    left[:, 4 * b:] = right[:, 4 * b:]
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


# consistency without a tie check and a wide left-right tolerance: nearly every pixel reaches the refinement
BASE = dict(nxcorr_threshold=0.5, consistency=True, max_lr_diff=4096, no_dupes=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [9, 17, 33, 12, 40, 65])  # exact stacks, and n below the compile-time capacity
@pytest.mark.parametrize("step", [0.1, 0.25, 0.3, 0.4])  # 21, 9, 7 and 6 steps
def test_screen_parity_on_near_ties(handle, oracles, n, step):
    left, right = _scene(n, 40, 160, seed=n * 10 + int(step * 10))
    _check(handle, oracles, left, right, dict(BASE, subpixel_step=step))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [9, 33, 40])
def test_screen_parity_at_min_variance_boundary(handle, oracles, n):
    """min_variance such that n * min_variance sits on the float variance (n - 1) / n of band 2, and on either side
    of it by a few units in the last place."""
    left, right = _scene(n, 40, 160, seed=7 + n)
    var = np.float32(n - 1) / np.float32(n)  # float var1 of a stack with var_n = n - 1, up to the chain's rounding
    for k in (-3, 0, 3):
        minvar_n = np.float32(var) * np.float32(1 + k * U)
        _check(handle, oracles, left, right, dict(BASE, subpixel_step=0.1, min_variance=float(minvar_n / n)))
    _check(handle, oracles, left, right, dict(BASE, subpixel_step=0.1, min_variance=0.0))


def test_scene_forces_more_than_two_candidates():
    """Band 3 of the scene is constant along the row: every step interpolates the same values, so all steps have
    the same exact score and the same screened score, and the kernel has to take its unscreened loop there."""
    left, right = _scene(33, 40, 160, seed=1)
    b = 40 // 5
    band = right[:, 3 * b:4 * b].astype(np.int64)
    assert (band == band[:, :, :1]).all()
    v = band[:, :, 0]
    assert (v.max(axis=0) > v.min(axis=0)).all(), "nonconstant stacks, so that the tied scores are numbers"
