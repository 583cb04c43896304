"""Seeded, counter-based synthetic stereo stacks (SURVEY.md section 8d).

Every pixel is a pure function of (seed, image index t, absolute row r, column c),
so the CPU oracle, the GPU and every row- or frame-shard produce identical data
without communicating. The same code runs on numpy arrays and on torch tensors
(``xp`` = the numpy module or the torch module): all arithmetic is done in int64
on values kept below 2**32, which wraps identically in both libraries.

Scene: the right image of shot t is a smooth (quadratic B-spline) random pattern
evaluated on a 2x oversampled column grid; the left image samples the same pattern shifted by the
true disparity d(r, c) (a multiple of 0.5 px), then both sides get independent
integer noise in [-3, 3] (scaled for 16-bit). Special row bands exercise the
reference's edge cases: a low-contrast band (min_variance), a band with an exactly
periodic right row (NODUPES ties), a saturated band (wrap-around in the subpixel
interpolation) and disparities that point outside the right image.

The reference bench seed is 0x600DF00D (reference bench/cuda.cu:39).
"""

from __future__ import annotations

import numpy as np

DEFAULT_SEED = 0x600DF00D
_M32 = 0xFFFFFFFF


def _mix(x):
    """32-bit avalanche on int64 lanes holding values < 2**32."""
    x = x ^ (x >> 15)
    x = (x * 0x2C1B3C6D) & _M32
    x = x ^ (x >> 12)
    x = (x * 0x297A2D39) & _M32
    x = x ^ (x >> 15)
    return x


def _hash(seed, t, r, k):
    """hash(seed, t, r, k) -> int64 in [0, 2**32); t, r, k broadcastable integer arrays (k may be negative)."""
    x = (t * 0x9E3779B1 + 0x7F4A7C15) & _M32
    x = _mix(x ^ (seed & _M32))
    x = _mix((x + r * 0x85EBCA77) & _M32)
    x = _mix((x + ((k + 0x10000) & _M32) * 0xC2B2AE3D) & _M32)
    return x


def true_disparity_x2(r, c, width):
    """Ground-truth disparity in half-pixel units for absolute rows r and columns c (int64 arrays)."""
    third = max(width // 3, 1)
    region = c // third
    d2 = 34 + 0 * (r + c)  # 17 px
    d2 = d2 + (region == 1) * (81 - 34)  # 40.5 px
    d2 = d2 + (region >= 2) * (126 - 34)  # 63 px
    # a slow ramp on every other 64-row block: +0.5 px every 16 columns
    ramp = ((r // 64) % 2 == 1) * ((c // 16) % 24)
    return d2 + ramp


def make_stacks(n, height, width, dtype=np.uint8, seed=DEFAULT_SEED, row0=0, rows=None,
                frame=0, xp=np, device=None, bands=True):
    """Return (stack0, stack1, disp_true) with stack shapes [n, rows, width].

    stack0 is the left stack, stack1 the right stack; disp_true is float32 [rows, width]
    (left pixel (r, c) corresponds to right column c - disp_true). ``row0``/``rows`` select
    a row block of the full ``height`` x ``width`` scene; ``frame`` decorrelates frames of a batch.
    """
    if rows is None:
        rows = height - row0
    is16 = np.dtype(dtype) == np.uint16
    if not is16 and np.dtype(dtype) != np.uint8:
        raise ValueError("dtype must be uint8 or uint16")
    vmask = 0xFFF if is16 else 0xFF
    vshift = 4 if is16 else 0
    vmax = 65535 if is16 else 255
    noise_amp = 3 << vshift

    if xp is np:
        def arange(m):
            return np.arange(m, dtype=np.int64)

        def where(cnd, a, b):
            return np.where(cnd, a, b)

        def clip(a, lo, hi):
            return np.clip(a, lo, hi)

        def cast(a):
            return a.astype(dtype)

        def tofloat(a):
            return a.astype(np.float32)
    else:
        torch = xp

        def arange(m):
            return torch.arange(m, dtype=torch.int64, device=device)

        def where(cnd, a, b):
            return torch.where(cnd, a, b)

        def clip(a, lo, hi):
            return torch.clamp(a, lo, hi)

        tdt = torch.uint16 if is16 else torch.uint8

        def cast(a):
            return a.to(torch.int32).to(tdt) if is16 else a.to(tdt)

        def tofloat(a):
            return a.to(torch.float32)

    seed = (int(seed) + 0x51ED27 * int(frame)) & _M32
    t = arange(n).reshape(n, 1, 1)
    r = (arange(rows) + int(row0)).reshape(1, rows, 1)
    c = arange(width).reshape(1, 1, width)

    d2 = true_disparity_x2(r, c, width)  # [1, rows, width]

    band = (r // 32) % 16 if bands else r * 0 - 1
    is_low = band == 5  # low contrast
    is_dup = band == 9  # periodic right row, no noise
    is_sat = band == 13  # saturated
    period2 = 2 * 48  # duplicate period: 48 px

    def pattern(k):
        # band-limited sample at half-sample index k: quadratic B-spline over a coarse
        # random grid with a pitch of 8 half-samples (4 px); integer weights sum to 128
        kk = where(is_dup, k % period2, k)
        q = kk >> 3
        f = kk & 7
        w0 = (8 - f) * (8 - f)
        w2 = f * f
        w1 = 128 - w0 - w2
        u0 = _hash(seed, t, r, q) & vmask
        u1 = _hash(seed, t, r, q + 1) & vmask
        u2 = _hash(seed, t, r, q + 2) & vmask
        return ((w0 * u0 + w1 * u1 + w2 * u2 + 64) >> 7) << vshift

    right = pattern(2 * c)
    left = pattern(2 * c - d2)

    nz_r = (_hash(seed ^ 0xA5A5A5A5, t, r, c) % (2 * noise_amp + 1)) - noise_amp
    nz_l = (_hash(seed ^ 0x5A5A5A5A, t, r, c) % (2 * noise_amp + 1)) - noise_amp
    nz_r = where(is_dup, nz_r * 0, nz_r)

    # low-contrast band: constant 100 +- 1 (scaled)
    low_r = (100 << vshift) + (_hash(seed ^ 0x0F0F0F0F, t, r, c) % 3) - 1
    low_l = (100 << vshift) + (_hash(seed ^ 0xF0F0F0F0, t, r, c) % 3) - 1

    right = right + nz_r
    left = left + nz_l
    # saturated band: gain 3 then clamp, so long runs sit at vmax next to dark pixels
    right = where(is_sat, right * 3 - (vmax // 2), right)
    left = where(is_sat, left * 3 - (vmax // 2), left)
    right = where(is_low, low_r, right)
    left = where(is_low, low_l, left)

    right = cast(clip(right, 0, vmax))
    left = cast(clip(left, 0, vmax))
    disp = tofloat(d2[0]) * 0.5
    return left, right, disp


def random_stacks(n, height, width, dtype=np.uint8, seed=1):
    """Fully random, uncorrelated stacks (many ties / no true match) for stage-level tests."""
    rng = np.random.default_rng(seed)
    hi = 65536 if np.dtype(dtype) == np.uint16 else 256
    a = rng.integers(0, hi, size=(n, height, width), dtype=np.int64).astype(dtype)
    b = rng.integers(0, hi, size=(n, height, width), dtype=np.int64).astype(dtype)
    return a, b


def rectify_maps(rows, cols, src_rows=None, src_cols=None, camera=0, k1=-0.12, k2=0.03, angle_deg=0.6):
    """Float32 rectification maps (map_x, map_y) [rows, cols] of a pinhole camera with radial distortion (k1, k2)
    and a small rotation about the optical axis and the vertical axis, what cv2.initUndistortRectifyMap(K, D, R, P,
    (cols, rows), CV_32FC1) computes: for a rectified pixel (u, v), the ray R^-1 P^-1 (u, v, 1), projected and
    distorted into the source image of src_rows x src_cols (default: the rectified size). camera = 0 / 1 mirrors the
    rotation, as the two cameras of a rig are rotated towards each other."""
    src_rows = rows if src_rows is None else src_rows
    src_cols = cols if src_cols is None else src_cols
    f = 0.9 * max(src_rows, src_cols)
    cx, cy = (src_cols - 1) / 2.0, (src_rows - 1) / 2.0
    fn = 0.9 * max(rows, cols)  # P: the rectified camera
    cxn, cyn = (cols - 1) / 2.0, (rows - 1) / 2.0
    a = np.deg2rad(angle_deg) * (1 if camera == 0 else -1)
    rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    b = 2 * a
    ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    rinv = (rz @ ry).T
    v, u = np.mgrid[0:rows, 0:cols].astype(np.float64)
    ray = np.stack([(u - cxn) / fn, (v - cyn) / fn, np.ones_like(u)], axis=-1) @ rinv.T
    x, y = ray[..., 0] / ray[..., 2], ray[..., 1] / ray[..., 2]
    r2 = x * x + y * y
    radial = 1 + k1 * r2 + k2 * r2 * r2
    return (f * x * radial + cx).astype(np.float32), (f * y * radial + cy).astype(np.float32)
