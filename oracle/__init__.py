"""CPU checkers for the BICOS::match hot path. TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this package. Nothing under libbicos_b200/ does: the product path
is CUDA-only and fails loudly without its extension.

Two checkers, same Python surface:

* ``oracle.ref``  -- the UNMODIFIED reference CPU backend (<REFERENCE_DIR>/src/impl/cpu.cpp
  and friends) compiled against oracle/shim into oracle/_ref/libbicos_ref.so by
  oracle/Makefile when BICOS_REFERENCE_DIR names a checkout of the reference project (a prebuilt
  oracle/_ref is kept otherwise); ``oracle.ref.available()`` says whether it can be loaded.
* ``oracle.port`` -- oracle/bicos_oracle.c, a plain-C restatement of the same algorithm
  (each function cites the reference file:line it follows). Pinned against ``oracle.ref``
  and against tests/golden/*.npz (generated from ``oracle.ref`` by tests/golden/make_golden.py); without the
  reference build, the tests that compare with it use the outputs stored under tests/golden/reference/
  (tests/golden/make_reference_outputs.py).
"""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# a checkout of the reference project, whose sources oracle/Makefile compiles into oracle/_ref
REFERENCE_DIR = os.environ.get("BICOS_REFERENCE_DIR", "")


def reference_sources_present() -> bool:
    return bool(REFERENCE_DIR) and os.path.exists(os.path.join(REFERENCE_DIR, "src", "impl", "cpu.cpp"))

CV_8U, CV_16U, CV_16S, CV_32F, CV_64F = 0, 2, 3, 5, 6
FLAG_NODUPES, FLAG_CONSISTENCY = 1, 2
INVALID_I16 = -32768


def build(ref: bool = True) -> None:
    """Compile the checkers (make is incremental). Building the checker is not using it."""
    targets = ["port"] + (["ref"] if ref else [])
    subprocess.run(["make", "-s", "-C", _HERE] + targets, check=True)


def _depth(a: np.ndarray) -> int:
    if a.dtype == np.uint8:
        return CV_8U
    if a.dtype == np.uint16:
        return CV_16U
    raise ValueError("stacks must be uint8 or uint16")


def _c(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a)


def _p(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def _opt(v) -> float:
    return -1.0 if v is None else float(v)


MODE_WIDE = 2  # bit 1 of the `mode` ints: allow the 384 / 512-bit extension (FULL, 17..23 images)


def _mode(mode_full, wide) -> int:
    return int(bool(mode_full)) | (MODE_WIDE if wide else 0)


def words_per_descriptor(n: int, full: bool, wide: bool = False) -> int:
    """Descriptor width choice of the reference driver (src/impl/cpu.cpp:122-156); `wide` adds the
    12- and 16-word descriptors of this repository's extension."""
    bits = n * n - 2 * n + 3 if full else 4 * n - 7
    for k, cap in ((1, 32), (2, 64), (4, 128), (8, 256)) + (((12, 384), (16, 512)) if wide else ()):
        if bits <= cap:
            return k
    raise ValueError(f"input stacks too large, would require {bits} bits")


class _Lib:
    """Shared ctypes surface of libbicos_ref.so (prefix 'ref_') and libbicos_oracle.so (prefix 'orc_')."""

    def __init__(self, path: str, prefix: str, has_double: bool):
        self.path = path
        self.prefix = prefix
        self.has_double = has_double
        self._lib = None

    def available(self) -> bool:
        return os.path.exists(self.path)

    @property
    def lib(self):
        if self._lib is None:
            if not self.available():
                raise RuntimeError(f"{self.path} missing: run `make -C oracle`")
            lib = ctypes.CDLL(self.path)
            f = getattr(lib, self.prefix + "last_error")
            f.restype = ctypes.c_char_p
            getattr(lib, self.prefix + "hardware_threads").restype = ctypes.c_int
            self._lib = lib
        return self._lib

    def _fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def _check(self, rc):
        if rc < 0:
            raise RuntimeError(self._fn("last_error")().decode())
        return rc

    def set_threads(self, n: int) -> None:
        self._fn("set_threads")(ctypes.c_int(n))

    def hardware_threads(self) -> int:
        return int(self._fn("hardware_threads")())

    # -- full path -------------------------------------------------------------------------
    def match(self, stack0, stack1, nxcorr_threshold=0.5, subpixel_step=None, min_variance=None,
              mode_full=False, consistency=False, max_lr_diff=1, no_dupes=False, double=False, wide_descriptors=False):
        """BICOS::match on planar [n, H, W] stacks. Returns (disparity, corrmap or None).

        ``wide_descriptors`` (extension, same name as in BICOS::Config): descriptors of 384 / 512 bits. The port handles them in its own driver;
        for the reference build, whose driver throws above 256 bits (src/impl/cpu.cpp:153-155), the
        path is composed here from the reference's own stage templates instantiated with
        std::bitset<384> / <512> (descriptor_transform -> bicos -> agree, the sequence of
        match_impl, src/impl/cpu.cpp:35-98)."""
        s0, s1 = _c(stack0), _c(stack1)
        n, rows, cols = s0.shape
        if wide_descriptors and self.prefix == "ref_" and words_per_descriptor(n, mode_full, True) > 8:
            return self._match_by_stages(s0, s1, nxcorr_threshold, subpixel_step, min_variance, mode_full,
                                         consistency, max_lr_diff, no_dupes)
        disp_buf = np.empty((rows, cols), dtype=np.float32)
        disp_type = ctypes.c_int(-1)
        if double:
            if not self.has_double:
                raise RuntimeError("the reference CPU backend has no double path")
            corr = np.full((rows, cols), np.nan, dtype=np.float64)
            fn = self._fn("match_f64")
        else:
            corr = np.full((rows, cols), np.nan, dtype=np.float32)
            fn = self._fn("match")
        rc = fn(_p(s0), _p(s1), ctypes.c_int(n), ctypes.c_int(rows), ctypes.c_int(cols),
                ctypes.c_int(_depth(s0)), ctypes.c_float(_opt(nxcorr_threshold)),
                ctypes.c_float(_opt(subpixel_step)), ctypes.c_float(_opt(min_variance)),
                ctypes.c_int(_mode(mode_full, wide_descriptors)), ctypes.c_int(int(consistency)),
                ctypes.c_int(int(max_lr_diff)), ctypes.c_int(int(no_dupes)),
                _p(disp_buf), ctypes.byref(disp_type), _p(corr))
        self._check(rc)
        if disp_type.value == CV_16S:
            disp = disp_buf.view(np.int16).reshape(-1)[: rows * cols].reshape(rows, cols).copy()
        else:
            disp = disp_buf
        return disp, (corr if nxcorr_threshold is not None else None)

    def _match_by_stages(self, s0, s1, nxcorr_threshold, subpixel_step, min_variance, mode_full,
                         consistency, max_lr_diff, no_dupes):
        d0 = self.descriptors(s0, mode_full, wide=True)
        d1 = self.descriptors(s1, mode_full, wide=True)
        flags = (FLAG_CONSISTENCY | (FLAG_NODUPES if no_dupes else 0)) if consistency else FLAG_NODUPES  # cpu.cpp:68-75
        raw = self.bicos(d0, d1, flags, max_lr_diff if consistency else -1)
        if nxcorr_threshold is None:
            return raw, None
        disp, corr = self.agree(raw, s0, s1, nxcorr_threshold, subpixel_step, min_variance)
        if subpixel_step is None:
            disp = disp.astype(np.float32)  # cpu.cpp:88-94: convertTo keeps -32768 as -32768.0f
        # cpu.cpp:78-81: the map starts as NaN; agree() of the harness does the same
        return disp, corr

    # -- stages ----------------------------------------------------------------------------
    def descriptors(self, stack, mode_full=False, wide=False):
        """[H, W, K] uint32 words, bit i of the descriptor = bit i%32 of word i//32."""
        s = _c(stack)
        n, rows, cols = s.shape
        out = np.zeros((rows, cols, 16), dtype=np.uint32)
        k = self._check(self._fn("descriptors")(
            _p(s), ctypes.c_int(n), ctypes.c_int(rows), ctypes.c_int(cols), ctypes.c_int(_depth(s)),
            ctypes.c_int(_mode(mode_full, wide)), _p(out), ctypes.c_int(16)))
        # the C side packs K words per pixel densely
        return out.reshape(-1)[: rows * cols * k].reshape(rows, cols, k).copy()

    def bicos(self, desc0, desc1, flags, max_lr_diff=-1):
        """Search + postfilter on [H, W, K] uint32 descriptors -> int16 [H, W] raw disparity."""
        d0, d1 = _c(desc0.astype(np.uint32, copy=False)), _c(desc1.astype(np.uint32, copy=False))
        rows, cols, k = d0.shape
        out = np.empty((rows, cols), dtype=np.int16)
        self._check(self._fn("bicos")(_p(d0), _p(d1), ctypes.c_int(k), ctypes.c_int(rows),
                                      ctypes.c_int(cols), ctypes.c_int(flags),
                                      ctypes.c_int(max_lr_diff), _p(out)))
        return out

    def agree(self, raw_disp, stack0, stack1, nxcorr_threshold, subpixel_step=None,
              min_variance=None, double=False):
        """Refine a raw int16 disparity. Returns (disparity int16|float32, corrmap).

        ``min_variance`` is the user-level value (multiplied by n here, like src/impl/cpu.cpp:127).
        """
        s0, s1 = _c(stack0), _c(stack1)
        raw = _c(raw_disp.astype(np.int16, copy=False))
        n, rows, cols = s0.shape
        di = np.empty((rows, cols), dtype=np.int16)
        df = np.empty((rows, cols), dtype=np.float32)
        mv = -1.0 if min_variance is None else float(np.float32(min_variance) * np.float32(n))
        if double:
            if not self.has_double:
                raise RuntimeError("the reference CPU backend has no double path")
            corr = np.empty((rows, cols), dtype=np.float64)
            fn = self._fn("agree_f64")
        else:
            corr = np.empty((rows, cols), dtype=np.float32)
            fn = self._fn("agree")
        self._check(fn(_p(raw), _p(s0), _p(s1), ctypes.c_int(n), ctypes.c_int(rows),
                       ctypes.c_int(cols), ctypes.c_int(_depth(s0)),
                       ctypes.c_float(float(nxcorr_threshold)), ctypes.c_float(_opt(subpixel_step)),
                       ctypes.c_float(mv), _p(di), _p(df), _p(corr)))
        return (di if subpixel_step is None else df), corr


ref = _Lib(os.path.join(_HERE, "_ref", "libbicos_ref.so"), "ref_", has_double=False)
port = _Lib(os.path.join(_HERE, "libbicos_oracle.so"), "orc_", has_double=True)


class _RefConfig(ctypes.Structure):
    _fields_ = [("nxcorr_threshold", ctypes.c_float), ("subpixel_step", ctypes.c_float),
                ("min_variance", ctypes.c_float), ("mode", ctypes.c_int), ("precision", ctypes.c_int),
                ("variant_type", ctypes.c_int), ("max_lr_diff", ctypes.c_int), ("no_dupes", ctypes.c_int)]


class _RefCuda:
    """The UNMODIFIED reference CUDA backend (src/impl/cuda.cu), compiled for sm_100a against
    oracle/shim by `make -C oracle refcuda` into oracle/_ref/libbicos_refcuda.so: the second
    baseline ("the reference's own CUDA build on the same B200"). Needs a GPU to run; used by
    bench.py / tools/bench_configs.py for timing and by one GPU test as a cross-check.

    Its outputs follow the reference's CUDA conventions, which differ from the CPU oracle:
    integer mode returns int16, corrmap cells that were never evaluated are uninitialised,
    and nvcc contracts the interpolation polynomial into FMAs (SURVEY.md 9.5)."""

    def __init__(self, path):
        self.path = path
        self._lib = None

    def available(self) -> bool:
        return os.path.exists(self.path)

    @property
    def lib(self):
        if self._lib is None:
            if not self.available():
                raise RuntimeError(f"{self.path} missing: run `make -C oracle refcuda`")
            self._lib = ctypes.CDLL(self.path)
            self._lib.refcuda_last_error.restype = ctypes.c_char_p
        return self._lib

    @staticmethod
    def _cfg(nxcorr_threshold=0.5, subpixel_step=None, min_variance=None, mode_full=False,
             consistency=False, max_lr_diff=1, no_dupes=False, double=False):
        return _RefConfig(_opt(nxcorr_threshold), _opt(subpixel_step), _opt(min_variance), int(mode_full),
                          int(double), int(consistency), int(max_lr_diff), int(no_dupes))

    def match(self, stack0, stack1, **kw):
        s0, s1 = _c(stack0), _c(stack1)
        n, rows, cols = s0.shape
        cfg = self._cfg(**kw)
        disp_buf = np.empty((rows, cols), dtype=np.float32)
        corr_buf = np.full((rows, cols), np.nan, dtype=np.float64)
        dt, ct = ctypes.c_int(0), ctypes.c_int(0)
        rc = self.lib.refcuda_match(_p(s0), _p(s1), ctypes.c_int(n), ctypes.c_int(rows), ctypes.c_int(cols),
                                    ctypes.c_int(_depth(s0)), ctypes.byref(cfg), _p(disp_buf), ctypes.byref(dt),
                                    _p(corr_buf), ctypes.byref(ct))
        if rc != 0:
            raise RuntimeError(self.lib.refcuda_last_error().decode())
        if dt.value == CV_16S:
            disp = disp_buf.view(np.int16).reshape(-1)[: rows * cols].reshape(rows, cols).copy()
        else:
            disp = disp_buf
        corr = None
        if ct.value == CV_32F:
            corr = corr_buf.view(np.float32).reshape(-1)[: rows * cols].reshape(rows, cols).copy()
        elif ct.value == CV_64F:
            corr = corr_buf
        return disp, corr

    def time(self, stack0, stack1, warmup=3, iters=10, **kw):
        """(median, min) ms per BICOS::match over `iters` individually timed calls, device-resident inputs."""
        s0, s1 = _c(stack0), _c(stack1)
        n, rows, cols = s0.shape
        cfg = self._cfg(**kw)
        med, mn = ctypes.c_float(0), ctypes.c_float(0)
        rc = self.lib.refcuda_time(_p(s0), _p(s1), ctypes.c_int(n), ctypes.c_int(rows), ctypes.c_int(cols),
                                   ctypes.c_int(_depth(s0)), ctypes.byref(cfg), ctypes.c_int(warmup),
                                   ctypes.c_int(iters), ctypes.byref(med), ctypes.byref(mn))
        if rc != 0:
            raise RuntimeError(self.lib.refcuda_last_error().decode())
        return float(med.value), float(mn.value)


refcuda = _RefCuda(os.path.join(_HERE, "_ref", "libbicos_refcuda.so"))
