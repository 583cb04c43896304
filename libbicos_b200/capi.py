"""ctypes binding of include/bicos_b200.h for callers that hold device memory in torch tensors.

PyTorch is plumbing here (allocation, streams, torch.distributed); every computation on the
path happens inside libbicos_b200.so. There is no fallback: if the shared library is missing
or no CUDA device is present, the calls raise.
"""

from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libbicos_b200.so")

DEPTH_8U, DEPTH_16U, TYPE_16S, TYPE_32F, TYPE_64F = 0, 2, 3, 5, 6
FLAG_NODUPES, FLAG_CONSISTENCY, FLAG_TOP_BIT_FREE, FLAG_TOP2_BITS_FREE = 1, 2, 4, 8
REPROJECT_ALLOW_NEGATIVE_Z = 1
MAX_IMAGES = 65

EXPORTS = (
    "bicos_b200_last_error", "bicos_b200_device_count", "bicos_b200_create", "bicos_b200_destroy",
    "bicos_b200_descriptor_words", "bicos_b200_disparity_type", "bicos_b200_corrmap_type",
    "bicos_b200_transform", "bicos_b200_search", "bicos_b200_search_range", "bicos_b200_refine", "bicos_b200_match",
    "bicos_b200_match_batch", "bicos_b200_set_overlap", "bicos_b200_match_host", "bicos_b200_match_host_begin", "bicos_b200_match_host_end", "bicos_b200_match_rows", "bicos_b200_synchronize",
    "bicos_b200_kernel_launches", "bicos_b200_set_profiling", "bicos_b200_stage_times",
    "bicos_b200_shared_alloc", "bicos_b200_shared_open", "bicos_b200_shared_close", "bicos_b200_shared_free",
    "bicos_b200_set_search_engine", "bicos_b200_get_search_engine", "bicos_b200_last_search_kernel",
    "bicos_b200_remap", "bicos_b200_match_rectified", "bicos_b200_reproject", "bicos_b200_filter_speckles",
    "bicos_b200_search_windows", "bicos_b200_match_windows", "bicos_b200_windows_from_disparity",
)
SEARCH_ENGINES = {"auto": 0, "popc": 1, "tensor": 2}
IPC_HANDLE_BYTES = 64


class BicosError(RuntimeError):
    """Raised for every non-zero status of the C ABI (BICOS::Exception in the reference)."""


class CConfig(ctypes.Structure):
    """bicos_b200_config == the reference's BicosConfig (src/pybicos_c.cpp:30-41)."""

    _fields_ = [
        ("nxcorr_threshold", ctypes.c_float),
        ("subpixel_step", ctypes.c_float),
        ("min_variance", ctypes.c_float),
        ("mode", ctypes.c_int),
        ("precision", ctypes.c_int),
        ("variant_type", ctypes.c_int),
        ("max_lr_diff", ctypes.c_int),
        ("no_dupes", ctypes.c_int),
        ("negative_threshold_is_set", ctypes.c_int),  # extension, see include/bicos_b200.h
        ("wide_descriptors", ctypes.c_int),  # extension: 384 / 512-bit descriptors (FULL, 17..23 images)
        ("has_disparity_range", ctypes.c_int),  # extension: search only min_disparity <= x_left - x_right <= max_disparity
        ("min_disparity", ctypes.c_int),
        ("max_disparity", ctypes.c_int),
    ]


@dataclass
class Config:
    """Python mirror of BICOS::Config (reference include/common.hpp:73-82)."""

    nxcorr_threshold: Optional[float] = 0.5
    subpixel_step: Optional[float] = None
    min_variance: Optional[float] = None
    mode_full: bool = False  # TransformMode::FULL
    double: bool = False  # Precision::DOUBLE
    consistency: bool = False  # Variant::Consistency instead of Variant::NoDuplicates
    max_lr_diff: int = 1
    no_dupes: bool = False
    wide_descriptors: bool = False  # extension beyond the reference: FULL stacks of 17..23 images
    # extension beyond the reference: (min, max), both inclusive, of x_left - x_right; None = the whole row.
    # See BICOS::Config::disparity_range.
    disparity_range: Optional[Tuple[int, int]] = None

    def to_c(self) -> CConfig:
        def opt(v):
            return -1.0 if v is None else float(v)

        negative = self.nxcorr_threshold is not None and not self.nxcorr_threshold >= 0
        rng = self.disparity_range
        return CConfig(opt(self.nxcorr_threshold), opt(self.subpixel_step), opt(self.min_variance),
                       int(self.mode_full), int(self.double), int(self.consistency),
                       int(self.max_lr_diff), int(self.no_dupes), int(negative),
                       int(self.wide_descriptors), int(rng is not None),
                       int(rng[0]) if rng is not None else 0, int(rng[1]) if rng is not None else 0)

    @property
    def flags(self) -> int:
        if self.consistency:
            return FLAG_CONSISTENCY | (FLAG_NODUPES if self.no_dupes else 0)
        return FLAG_NODUPES


class CRectifyMaps(ctypes.Structure):
    """bicos_b200_rectify_maps."""

    _fields_ = [("map_x0", ctypes.c_void_p), ("map_y0", ctypes.c_void_p), ("map_x1", ctypes.c_void_p),
                ("map_y1", ctypes.c_void_p), ("map_pitch_bytes", ctypes.c_size_t)]


class CDisparityWindows(ctypes.Structure):
    """bicos_b200_disparity_windows."""

    _fields_ = [("min_disparity", ctypes.c_void_p), ("max_disparity", ctypes.c_void_p), ("pitch_bytes", ctypes.c_size_t)]


@dataclass
class RectifyMaps:
    """Rectification maps of both cameras for Handle.match_rectified: float32 CUDA tensors [rows, cols] with
    contiguous rows, all of one shape and row stride, e.g. the CV_32FC1 maps of cv2.initUndistortRectifyMap.
    map_x0 / map_y0 rectify stack0, map_x1 / map_y1 stack1."""

    map_x0: object
    map_y0: object
    map_x1: object
    map_y1: object


_lib = None


def lib():
    """The loaded libbicos_b200.so. Raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BicosError(
                f"{LIB_PATH} is missing: build it with `make -C libbicos_b200/csrc` "
                "(or __graft_entry__.build()); there is no CPU or PyTorch fallback")
        L = ctypes.CDLL(LIB_PATH)
        L.bicos_b200_last_error.restype = ctypes.c_char_p
        L.bicos_b200_set_search_engine.argtypes = [ctypes.c_int]
        L.bicos_b200_get_search_engine.argtypes = []
        L.bicos_b200_last_search_kernel.restype = ctypes.c_char_p
        L.bicos_b200_last_search_kernel.argtypes = []
        L.bicos_b200_kernel_launches.restype = ctypes.c_longlong
        L.bicos_b200_kernel_launches.argtypes = [ctypes.c_void_p]
        vp, i, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
        cfgp = ctypes.POINTER(CConfig)
        pp = ctypes.POINTER(ctypes.c_void_p)
        L.bicos_b200_create.argtypes = [ctypes.POINTER(vp), i]
        L.bicos_b200_destroy.argtypes = [vp]
        L.bicos_b200_descriptor_words.argtypes = [i, i]
        L.bicos_b200_disparity_type.argtypes = [cfgp]
        L.bicos_b200_corrmap_type.argtypes = [cfgp]
        L.bicos_b200_transform.argtypes = [vp, pp, i, i, i, sz, i, i, vp, sz, vp]
        L.bicos_b200_search.argtypes = [vp, vp, vp, i, i, i, sz, i, vp, vp, vp, vp, vp]
        L.bicos_b200_search_range.argtypes = [vp, vp, vp, i, i, i, sz, i, vp, vp, vp, vp, i, i, vp]
        L.bicos_b200_refine.argtypes = [vp, pp, pp, i, i, i, sz, i, cfgp, vp, vp, vp, vp, vp, vp, sz, vp, sz, vp]
        L.bicos_b200_match.argtypes = [vp, pp, pp, i, i, i, sz, i, cfgp, vp, sz, vp, sz, vp]
        L.bicos_b200_match_batch.argtypes = [vp, i, vp, vp, i, i, i, sz, i, cfgp, vp, sz, vp, sz, vp]
        L.bicos_b200_set_overlap.argtypes = [vp, i]
        L.bicos_b200_match_rows.argtypes = [vp, pp, pp, i, i, i, sz, i, cfgp, i, i, vp, sz, vp, sz, vp]
        L.bicos_b200_match_host.argtypes = [vp, pp, pp, i, i, i, i, cfgp, vp, vp]
        L.bicos_b200_match_host_begin.argtypes = [vp, pp, pp, i, i, i, i, cfgp, vp, vp]
        L.bicos_b200_match_host_end.argtypes = [vp]
        L.bicos_b200_shared_alloc.argtypes = [i, sz, ctypes.POINTER(ctypes.c_void_p), vp]
        L.bicos_b200_shared_open.argtypes = [i, vp, ctypes.POINTER(ctypes.c_void_p)]
        L.bicos_b200_shared_close.argtypes = [i, vp]
        L.bicos_b200_shared_free.argtypes = [i, vp]
        L.bicos_b200_synchronize.argtypes = [vp, vp]
        L.bicos_b200_set_profiling.argtypes = [vp, i]
        L.bicos_b200_remap.argtypes = [vp, pp, i, i, i, sz, i, vp, vp, sz, i, i, pp, sz, vp]
        L.bicos_b200_match_rectified.argtypes = [vp, pp, pp, i, i, i, sz, i, ctypes.POINTER(CRectifyMaps), i, i, cfgp, vp, sz, vp,
                                                 sz, vp]
        L.bicos_b200_reproject.argtypes = [vp, vp, i, sz, i, i, ctypes.POINTER(ctypes.c_double), i, vp, sz, vp, vp, vp, vp]
        L.bicos_b200_filter_speckles.argtypes = [vp, vp, i, sz, i, i, ctypes.c_double, i, ctypes.c_double, vp, vp]
        winp = ctypes.POINTER(CDisparityWindows)
        L.bicos_b200_search_windows.argtypes = [vp, vp, vp, i, i, i, sz, i, vp, vp, vp, vp, winp, vp]
        L.bicos_b200_match_windows.argtypes = [vp, pp, pp, i, i, i, sz, i, cfgp, winp, vp, sz, vp, sz, vp]
        L.bicos_b200_windows_from_disparity.argtypes = [vp, vp, i, sz, i, i, i, i, i, vp, vp, sz, vp]
        L.bicos_b200_stage_times.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]
        _lib = L
    return _lib


def _check(rc: int) -> int:
    if rc < 0:
        raise BicosError(lib().bicos_b200_last_error().decode())
    return rc


MODE_WIDE = 2  # BICOS_B200_MODE_WIDE


def descriptor_words(n: int, mode_full: bool = False, wide: bool = False) -> int:
    """Words per descriptor: 1/2/4/8 as the reference dispatches them; `wide` (extension) adds 12 / 16."""
    return _check(lib().bicos_b200_descriptor_words(n, int(mode_full) | (MODE_WIDE if wide else 0)))


def set_search_engine(engine: str) -> None:
    """'auto' (tensor cores where they apply), 'popc' or 'tensor': bicos_b200_set_search_engine, process-wide."""
    _check(lib().bicos_b200_set_search_engine(SEARCH_ENGINES[engine]))


def search_engine() -> str:
    code = lib().bicos_b200_get_search_engine()
    return next(k for k, v in SEARCH_ENGINES.items() if v == code)


def last_search_kernel() -> str:
    """Which kernel this thread's last search dispatched, e.g. 'mma2<K=4,nodupes=0,ct=1,dirs=2>' or 'popc<K=4,flags=2>'."""
    return lib().bicos_b200_last_search_kernel().decode()


def _ptr_array(ptrs: Sequence[int]):
    arr = (ctypes.c_void_p * len(ptrs))()
    for k, p in enumerate(ptrs):
        arr[k] = p
    return arr


class Handle:
    """Owns one per-device workspace (bicos_b200_handle)."""

    def __init__(self, device: Optional[int] = None):
        h = ctypes.c_void_p()
        _check(lib().bicos_b200_create(ctypes.byref(h), -1 if device is None else int(device)))
        self._h = h

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().bicos_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def kernel_launches(self) -> int:
        return int(lib().bicos_b200_kernel_launches(self._h))

    # ---- torch-tensor helpers -----------------------------------------------------------
    @staticmethod
    def _stack_info(stack):
        import torch

        if stack.dim() != 3 or not stack.is_cuda:
            raise BicosError("stacks must be CUDA tensors of shape [n, rows, cols]")
        if stack.dtype == torch.uint8:
            depth, eb = DEPTH_8U, 1
        elif stack.dtype == torch.uint16:
            depth, eb = DEPTH_16U, 2
        else:
            raise BicosError("bad input depths, only uint8 and uint16 are supported")
        if stack.stride(2) != 1:
            raise BicosError("stack rows must be contiguous")
        n, rows, cols = stack.shape
        pitch = stack.stride(1) * eb
        planes = _ptr_array([stack.data_ptr() + stack.stride(0) * eb * t for t in range(n)])
        return planes, n, rows, cols, pitch, depth

    @staticmethod
    def _stream():
        import torch

        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ---- stages -------------------------------------------------------------------------
    def transform(self, stack, mode_full: bool = False, wide: bool = False):
        """Descriptor transform of one stack -> int32 tensor [rows, cols, K] (a view of pitched rows)."""
        import torch

        planes, n, rows, cols, pitch, depth = self._stack_info(stack)
        k = descriptor_words(n, mode_full, wide)
        pitch_words = (cols * k + 3) // 4 * 4
        desc = torch.empty((rows, pitch_words), dtype=torch.int32, device=stack.device)
        _check(lib().bicos_b200_transform(self._h, planes, n, rows, cols, pitch, depth,
                                          int(mode_full) | (MODE_WIDE if wide else 0),
                                          desc.data_ptr(), pitch_words, self._stream()))
        return desc, k

    def search(self, desc0, desc1, k: int, cols: int, flags: int, top_bit_free=False, disparity_range=None, windows=None):
        """Row-wise search on pitched descriptors -> (fwd_first, fwd_last, rev_first, rev_last).

        Each is a [rows, cols] int32 tensor holding uint32 keys cost << 16 | column (see
        include/bicos_b200.h), or None when `flags` does not need it. ``top_bit_free``: the caller
        vouches that bit 32k-1 of every descriptor is zero (BICOS_B200_FLAG_TOP_BIT_FREE; true for
        transform() output), which lets the tensor-core engine use its column-term kernels; ``top_bit_free=2``: the
        top TWO bits are zero (BICOS_B200_FLAG_TOP2_BITS_FREE; also true for transform() output), which adds the
        one-pass consistency kernel. ``disparity_range`` = (min, max): only the pairs with min <= x_left - x_right <= max
        (bicos_b200_search_range); fwd_last is then always returned, and refine() needs a Config with the same range.
        ``windows`` = (min, max) int16 CUDA tensors [rows, cols]: per-pixel bounds instead (bicos_b200_search_windows);
        fwd_last is always returned, and refine() needs a Config with a range that does not cover the row, e.g. (0, 0)."""
        import torch

        rows, pitch_words = desc0.shape
        dev = desc0.device

        def keys(needed):
            return torch.empty((rows, cols), dtype=torch.int32, device=dev) if needed else None

        fwdf = keys(True)
        fwdl = keys(flags & FLAG_NODUPES or disparity_range is not None or windows is not None)
        revf = keys(flags & FLAG_CONSISTENCY)
        revl = keys(flags == (FLAG_NODUPES | FLAG_CONSISTENCY))
        ptr = [t.data_ptr() if t is not None else None for t in (fwdf, fwdl, revf, revl)]
        flags |= FLAG_TOP2_BITS_FREE if int(top_bit_free) >= 2 else FLAG_TOP_BIT_FREE if top_bit_free else 0
        if windows is not None:
            if disparity_range is not None:
                raise BicosError("disparity windows and a disparity range exclude each other")
            cw = self._windows_info(windows, rows, cols, dev)
            _check(lib().bicos_b200_search_windows(self._h, desc0.data_ptr(), desc1.data_ptr(), k, rows, cols, pitch_words, flags,
                                                   *ptr, ctypes.byref(cw), self._stream()))
        elif disparity_range is None:
            _check(lib().bicos_b200_search(self._h, desc0.data_ptr(), desc1.data_ptr(), k, rows, cols, pitch_words, flags,
                                           *ptr, self._stream()))
        else:
            _check(lib().bicos_b200_search_range(self._h, desc0.data_ptr(), desc1.data_ptr(), k, rows, cols, pitch_words, flags,
                                                 *ptr, int(disparity_range[0]), int(disparity_range[1]), self._stream()))
        return fwdf, fwdl, revf, revl

    def _outputs(self, cfg: Config, rows: int, cols: int, device):
        import torch

        ccfg = cfg.to_c()
        dt = lib().bicos_b200_disparity_type(ctypes.byref(ccfg))
        ct = lib().bicos_b200_corrmap_type(ctypes.byref(ccfg))
        disp = torch.empty((rows, cols), dtype=torch.int16 if dt == TYPE_16S else torch.float32, device=device)
        corr = None
        if ct:
            corr = torch.empty((rows, cols), dtype=torch.float64 if ct == TYPE_64F else torch.float32, device=device)
        return ccfg, disp, corr

    def refine(self, stack0, stack1, cfg: Config, keys, want_raw: bool = True):
        """Postfilter + NXC refinement on the 4-tuple returned by search()
        -> (disparity, corrmap or None, raw int16 or None)."""
        import torch

        p0, n, rows, cols, pitch, depth = self._stack_info(stack0)
        p1, n1, rows1, cols1, pitch1, depth1 = self._stack_info(stack1)
        if (n1, rows1, cols1, pitch1, depth1) != (n, rows, cols, pitch, depth):
            raise BicosError("stack0 and stack1 differ")
        ccfg, disp, corr = self._outputs(cfg, rows, cols, stack0.device)
        raw = torch.empty((rows, cols), dtype=torch.int16, device=stack0.device) if want_raw else None
        _check(lib().bicos_b200_refine(
            self._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg),
            *[t.data_ptr() if t is not None else None for t in keys],
            raw.data_ptr() if raw is not None else None, disp.data_ptr(), disp.stride(0) * disp.element_size(),
            corr.data_ptr() if corr is not None else None,
            corr.stride(0) * corr.element_size() if corr is not None else 0, self._stream()))
        return disp, corr, raw

    @staticmethod
    def _check_out(ccfg, out, rows: int, cols: int, device=None):
        """Caller-supplied (disparity, corrmap) buffers must have the types bicos_b200_disparity_type /
        _corrmap_type name for this configuration, shape (rows, cols) and unit inner stride: the kernels and
        the D2H copies write rows * cols elements of that type without looking at the buffer again.
        `device` = a torch device for the device-resident entry points, None for host (numpy) buffers,
        which must also be C-contiguous (they are filled by flat copies)."""
        import numpy as np

        dt = lib().bicos_b200_disparity_type(ctypes.byref(ccfg))
        ct = lib().bicos_b200_corrmap_type(ctypes.byref(ccfg))
        try:
            disp, corr = out
        except (TypeError, ValueError):
            raise BicosError("out must be a (disparity, corrmap) pair") from None
        want_np = {TYPE_16S: np.int16, TYPE_32F: np.float32, TYPE_64F: np.float64}

        def check(buf, code, what):
            if device is not None:
                import torch

                want = {TYPE_16S: torch.int16, TYPE_32F: torch.float32, TYPE_64F: torch.float64}[code]
                if not isinstance(buf, torch.Tensor) or buf.dtype != want:
                    raise BicosError(f"out {what} must be a {want} tensor for this configuration")
                if buf.device != device:
                    raise BicosError(f"out {what} lives on {buf.device}, the stacks on {device}")
                if tuple(buf.shape) != (rows, cols) or buf.stride(1) != 1 or buf.stride(0) < cols:
                    raise BicosError(f"out {what} must have shape ({rows}, {cols}) with contiguous rows")
            else:
                if not isinstance(buf, np.ndarray) or buf.dtype != want_np[code]:
                    raise BicosError(f"out {what} must be a {np.dtype(want_np[code]).name} array for this configuration")
                if buf.shape != (rows, cols) or not buf.flags.c_contiguous or not buf.flags.writeable:
                    raise BicosError(f"out {what} must be a writable C-contiguous array of shape ({rows}, {cols})")

        if disp is None:
            raise BicosError("out disparity is None")
        check(disp, dt, "disparity")
        if ct:
            if corr is None:
                raise BicosError("this configuration has a threshold: out needs a corrmap buffer")
            check(corr, ct, "corrmap")
        elif corr is not None:
            raise BicosError("this configuration has no threshold: out corrmap must be None")
        return disp, corr

    # ---- whole path ---------------------------------------------------------------------
    def match(self, stack0, stack1, cfg: Config, out=None, rows_range=None):
        """Device-resident BICOS::match on [n, rows, cols] uint8/uint16 CUDA tensors.

        ``out`` = (disparity, corrmap) tensors to reuse; ``rows_range`` = (begin, end) matches only
        those rows (row-sharding) and leaves the others of ``out`` untouched.
        """
        p0, n, rows, cols, pitch, depth = self._stack_info(stack0)
        p1, n1, rows1, cols1, pitch1, depth1 = self._stack_info(stack1)
        if (n1, rows1, cols1, pitch1, depth1) != (n, rows, cols, pitch, depth):
            raise BicosError("stack0 and stack1 differ")
        if out is None:
            ccfg, disp, corr = self._outputs(cfg, rows, cols, stack0.device)
        else:
            ccfg = cfg.to_c()
            disp, corr = self._check_out(ccfg, out, rows, cols, stack0.device)
        args = [disp.data_ptr(), disp.stride(0) * disp.element_size(),
                corr.data_ptr() if corr is not None else None,
                corr.stride(0) * corr.element_size() if corr is not None else 0, self._stream()]
        if rows_range is None:
            _check(lib().bicos_b200_match(self._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), *args))
        else:
            _check(lib().bicos_b200_match_rows(self._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg),
                                               int(rows_range[0]), int(rows_range[1]), *args))
        return disp, corr

    @staticmethod
    def _windows_info(windows, rows: int, cols: int, device) -> CDisparityWindows:
        """bicos_b200_disparity_windows of a (min, max) pair of int16 CUDA tensors [rows, cols] with one row stride."""
        import torch

        try:
            wmin, wmax = windows
        except (TypeError, ValueError):
            raise BicosError("windows must be a (min_disparity, max_disparity) pair") from None
        for m in (wmin, wmax):
            if not isinstance(m, torch.Tensor) or m.dtype != torch.int16 or m.dim() != 2 or not m.is_cuda:
                raise BicosError("disparity windows must be int16 CUDA tensors of shape [rows, cols]")
            if m.device != device:
                raise BicosError(f"a disparity window map lives on {m.device}, the stacks on {device}")
            if tuple(m.shape) != (rows, cols) or m.stride(1) != 1:
                raise BicosError(f"disparity window maps must have shape ({rows}, {cols}) with contiguous rows")
        if wmin.stride(0) != wmax.stride(0):
            raise BicosError("both disparity window maps must share one row stride")
        return CDisparityWindows(wmin.data_ptr(), wmax.data_ptr(), wmin.stride(0) * 2)

    def match_windows(self, stack0, stack1, windows, cfg: Config, out=None):
        """match() with the search bounded per pixel (bicos_b200_match_windows): ``windows`` = (min, max) int16 CUDA
        tensors [rows, cols]; left pixel (r, i) pairs with right column j iff min[r, i] <= i - j <= max[r, i], and
        min > max makes the pixel invalid without searching it. ``cfg.disparity_range`` must be None.
        ``out`` = (disparity, corrmap) tensors to reuse."""
        p0, n, rows, cols, pitch, depth = self._stack_info(stack0)
        p1, n1, rows1, cols1, pitch1, depth1 = self._stack_info(stack1)
        if (n1, rows1, cols1, pitch1, depth1) != (n, rows, cols, pitch, depth):
            raise BicosError("stack0 and stack1 differ")
        cw = self._windows_info(windows, rows, cols, stack0.device)
        if out is None:
            ccfg, disp, corr = self._outputs(cfg, rows, cols, stack0.device)
        else:
            ccfg = cfg.to_c()
            disp, corr = self._check_out(ccfg, out, rows, cols, stack0.device)
        _check(lib().bicos_b200_match_windows(
            self._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), ctypes.byref(cw), disp.data_ptr(),
            disp.stride(0) * disp.element_size(), corr.data_ptr() if corr is not None else None,
            corr.stride(0) * corr.element_size() if corr is not None else 0, self._stream()))
        return disp, corr

    def windows_from_disparity(self, prior, margin: int, fallback=None, out=None):
        """Window maps from a prior disparity (bicos_b200_windows_from_disparity): [rows, cols] int16 / float32 CUDA
        tensor -> (min, max) int16 tensors. A valid prior d gives [floor(d) - margin, ceil(d) + margin] clamped to int16;
        an invalid one (-32768, NaN, -32768.0 or +-inf) gives ``fallback`` = (min, max), None = the whole row.
        ``out`` = a (min, max) pair of int16 tensors [rows, cols] with one row stride to fill."""
        import torch

        code, rows, cols, pitch = self._disparity_info(prior)
        fb = (-32768, 32767) if fallback is None else (int(fallback[0]), int(fallback[1]))
        if out is None:
            out = (torch.empty((rows, cols), dtype=torch.int16, device=prior.device),
                   torch.empty((rows, cols), dtype=torch.int16, device=prior.device))
        cw = self._windows_info(out, rows, cols, prior.device)
        _check(lib().bicos_b200_windows_from_disparity(self._h, prior.data_ptr(), code, pitch, rows, cols, int(margin), fb[0], fb[1],
                                                       cw.min_disparity, cw.max_disparity, cw.pitch_bytes, self._stream()))
        return out

    @staticmethod
    def _map_info(maps, device):
        """(pointers, rows, cols, pitch in bytes) of float32 map tensors of one shape and row stride."""
        import torch

        first = maps[0]
        for m in maps:
            if not isinstance(m, torch.Tensor) or m.dtype != torch.float32 or m.dim() != 2 or not m.is_cuda:
                raise BicosError("rectification maps must be float32 CUDA tensors of shape [rows, cols]")
            if m.device != device:
                raise BicosError(f"a rectification map lives on {m.device}, the stacks on {device}")
            if m.shape != first.shape or m.stride() != first.stride() or m.stride(1) != 1:
                raise BicosError("rectification maps must share one shape and row stride, with contiguous rows")
        rows, cols = first.shape
        return [m.data_ptr() for m in maps], rows, cols, first.stride(0) * 4

    def remap(self, stack, map_x, map_y, out=None):
        """Rectification stage (bicos_b200_remap): [n, src_rows, src_cols] uint8 / uint16 CUDA tensor -> [n, rows, cols] of
        its dtype, out[i] = cv2.remap(stack[i], map_x, map_y, INTER_LINEAR, BORDER_CONSTANT, 0) bit for bit. ``map_x`` /
        ``map_y``: float32 CUDA tensors [rows, cols]. ``out``: a tensor of that shape and dtype, contiguous rows."""
        import torch

        planes, n, src_rows, src_cols, pitch, depth = self._stack_info(stack)
        (px, py), rows, cols, map_pitch = self._map_info([map_x, map_y], stack.device)
        if out is None:
            out = torch.empty((n, rows, cols), dtype=stack.dtype, device=stack.device)
        elif (not isinstance(out, torch.Tensor) or out.dtype != stack.dtype or tuple(out.shape) != (n, rows, cols)
              or out.device != stack.device):
            raise BicosError(f"out must be a {stack.dtype} tensor of shape ({n}, {rows}, {cols}) on {stack.device}")
        dst, _, _, _, dst_pitch, _ = self._stack_info(out)
        _check(lib().bicos_b200_remap(self._h, planes, n, src_rows, src_cols, pitch, depth, px, py, map_pitch, rows, cols,
                                      dst, dst_pitch, self._stream()))
        return out

    def match_rectified(self, stack0, stack1, maps: RectifyMaps, cfg: Config, out=None):
        """match() on raw stacks (bicos_b200_match_rectified): both stacks are remapped through ``maps`` into the
        handle's workspace (one launch), then matched; bit-identical to match(remap(stack0, ...), remap(stack1, ...)).
        The outputs have the maps' shape; ``out`` = (disparity, corrmap) tensors of that shape to reuse."""
        p0, n, src_rows, src_cols, pitch, depth = self._stack_info(stack0)
        p1, n1, rows1, cols1, pitch1, depth1 = self._stack_info(stack1)
        if (n1, rows1, cols1, pitch1, depth1) != (n, src_rows, src_cols, pitch, depth):
            raise BicosError("stack0 and stack1 differ")
        ptrs, rows, cols, map_pitch = self._map_info([maps.map_x0, maps.map_y0, maps.map_x1, maps.map_y1], stack0.device)
        if out is None:
            ccfg, disp, corr = self._outputs(cfg, rows, cols, stack0.device)
        else:
            ccfg = cfg.to_c()
            disp, corr = self._check_out(ccfg, out, rows, cols, stack0.device)
        cmaps = CRectifyMaps(*ptrs, map_pitch)
        _check(lib().bicos_b200_match_rectified(
            self._h, p0, p1, n, src_rows, src_cols, pitch, depth, ctypes.byref(cmaps), rows, cols, ctypes.byref(ccfg),
            disp.data_ptr(), disp.stride(0) * disp.element_size(), corr.data_ptr() if corr is not None else None,
            corr.stride(0) * corr.element_size() if corr is not None else 0, self._stream()))
        return disp, corr

    @staticmethod
    def _disparity_info(disparity):
        """(type code, rows, cols, pitch in bytes) of an int16 / float32 CUDA tensor [rows, cols] with contiguous rows."""
        import torch

        if not isinstance(disparity, torch.Tensor) or disparity.dim() != 2 or not disparity.is_cuda:
            raise BicosError("the disparity must be a CUDA tensor of shape [rows, cols]")
        codes = {torch.int16: TYPE_16S, torch.float32: TYPE_32F}
        if disparity.dtype not in codes:
            raise BicosError("the disparity must be int16 or float32")
        if disparity.stride(1) != 1:
            raise BicosError("disparity rows must be contiguous")
        rows, cols = disparity.shape
        return codes[disparity.dtype], rows, cols, disparity.stride(0) * disparity.element_size()

    @staticmethod
    def _q_matrix(Q):
        """Q as the 16 row-major float64 values the C ABI takes from host memory."""
        import numpy as np

        if hasattr(Q, "detach"):
            Q = Q.detach().cpu().numpy()
        q = np.ascontiguousarray(np.asarray(Q, dtype=np.float64))
        if q.shape != (4, 4):
            raise BicosError(f"Q must be 4 x 4, got shape {q.shape}")
        return (ctypes.c_double * 16)(*q.ravel().tolist())

    def reproject(self, disparity, Q, allow_negative_z: bool = False, out=None):
        """Dense reprojection (bicos_b200_reproject): [rows, cols] int16 / float32 CUDA disparity -> [rows, cols, 3]
        float32 X Y Z, NaN where a pixel is skipped (invalid disparity, non-finite point, Z < 0 unless
        ``allow_negative_z``); include/bicos_b200.h states the arithmetic. ``Q``: any 4 x 4 array-like. ``out``: a
        float32 tensor [rows, cols, 3] on the disparity's device with contiguous pixels."""
        import torch

        code, rows, cols, pitch = self._disparity_info(disparity)
        if out is None:
            out = torch.empty((rows, cols, 3), dtype=torch.float32, device=disparity.device)
        elif (not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or tuple(out.shape) != (rows, cols, 3)
              or out.device != disparity.device or out.stride(2) != 1 or out.stride(1) != 3):
            raise BicosError(f"out must be a float32 tensor of shape ({rows}, {cols}, 3) on {disparity.device} with contiguous rows")
        _check(lib().bicos_b200_reproject(self._h, disparity.data_ptr(), code, pitch, rows, cols, self._q_matrix(Q),
                                          REPROJECT_ALLOW_NEGATIVE_Z if allow_negative_z else 0, out.data_ptr(), out.stride(0) * 4,
                                          None, None, None, self._stream()))
        return out

    def reproject_points(self, disparity, Q, allow_negative_z: bool = False):
        """The kept points of reproject() in row-major pixel order -> (points [N, 3] float32, pixel_index [N] int32 =
        row * cols + col, counts), counts = {"points", "invalid_disparity", "non_finite", "negative_z"} summing to
        rows * cols. Synchronises the current stream to learn N; the tensors are views of rows * cols capacity."""
        import torch

        code, rows, cols, pitch = self._disparity_info(disparity)
        dev = disparity.device
        points = torch.empty((rows * cols, 3), dtype=torch.float32, device=dev)
        index = torch.empty((rows * cols,), dtype=torch.int32, device=dev)
        counts = torch.empty((4,), dtype=torch.int64, device=dev)
        _check(lib().bicos_b200_reproject(self._h, disparity.data_ptr(), code, pitch, rows, cols, self._q_matrix(Q),
                                          REPROJECT_ALLOW_NEGATIVE_Z if allow_negative_z else 0, None, 0, points.data_ptr(),
                                          index.data_ptr(), counts.data_ptr(), self._stream()))
        kept, invalid, non_finite, negative_z = (int(v) for v in counts.cpu().tolist())
        return points[:kept], index[:kept], dict(points=kept, invalid_disparity=invalid, non_finite=non_finite,
                                                 negative_z=negative_z)

    def filter_speckles(self, disparity, new_value, max_speckle_size: int, max_diff, counts: bool = False):
        """Speckle removal in place (bicos_b200_filter_speckles, cv::filterSpeckles' parameters in its order) on a
        [rows, cols] int16 / float32 CUDA disparity: every connected blob of at most ``max_speckle_size`` valid pixels
        whose 4-neighbours differ by at most ``max_diff`` is set to ``new_value``; include/bicos_b200.h states the
        semantics. Returns the tensor, or with ``counts`` (tensor, {"pixels", "speckles"}): the pixels set and the
        speckles removed, which synchronises the current stream. Without ``counts`` nothing synchronises."""
        import torch

        code, rows, cols, pitch = self._disparity_info(disparity)
        dev_counts = torch.empty((2,), dtype=torch.int64, device=disparity.device) if counts else None
        _check(lib().bicos_b200_filter_speckles(self._h, disparity.data_ptr(), code, pitch, rows, cols, float(new_value),
                                                int(max_speckle_size), float(max_diff),
                                                dev_counts.data_ptr() if counts else None, self._stream()))
        if not counts:
            return disparity
        pixels, speckles = (int(v) for v in dev_counts.cpu().tolist())
        return disparity, dict(pixels=pixels, speckles=speckles)

    def match_batch(self, frames, cfg: Config, outs=None):
        """Throughput mode (bicos_b200_match_batch): `frames` = [(stack0, stack1), ...] of one shape and dtype,
        device-resident; returns [(disparity, corrmap), ...]. Frame f + 1's transform + search run beside frame f's
        refine on two internal streams; the current stream is joined before and after."""
        if not frames:
            return []
        infos = [(self._stack_info(a), self._stack_info(b)) for a, b in frames]
        first = infos[0][0][1:]
        for ia, ib in infos:
            if ia[1:] != first or ib[1:] != first:
                raise BicosError("all stacks of a batch must agree in length, size, type and pitch")
        _, n, rows, cols, pitch, depth = infos[0][0]
        device = frames[0][0].device
        ccfg = cfg.to_c()
        if outs is None:
            outs = [self._outputs(cfg, rows, cols, device)[1:] for _ in frames]
        else:
            if len(outs) != len(frames):
                raise BicosError("outs must hold one (disparity, corrmap) pair per frame")
            outs = [self._check_out(ccfg, o, rows, cols, device) for o in outs]
        count = len(frames)
        p0 = (ctypes.c_void_p * count)(*[ctypes.cast(ia[0], ctypes.c_void_p) for ia, _ in infos])
        p1 = (ctypes.c_void_p * count)(*[ctypes.cast(ib[0], ctypes.c_void_p) for _, ib in infos])
        disp = (ctypes.c_void_p * count)(*[d.data_ptr() for d, _ in outs])
        has_corr = outs[0][1] is not None
        corr = (ctypes.c_void_p * count)(*[c.data_ptr() for _, c in outs]) if has_corr else None
        d0, c0 = outs[0]
        for d, c in outs:
            if d.stride(0) != d0.stride(0) or (has_corr and c.stride(0) != c0.stride(0)):
                raise BicosError("all outputs of a batch must share one pitch")
        _check(lib().bicos_b200_match_batch(
            self._h, count, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), disp, d0.stride(0) * d0.element_size(),
            corr, c0.stride(0) * c0.element_size() if has_corr else 0, self._stream()))
        self._batch_keepalive = (infos, p0, p1, disp, corr)
        return list(outs)

    def match_raw(self, stack0, stack1, cfg: Config, disp_ptr: int, disp_pitch: int, corr_ptr: Optional[int],
                  corr_pitch: int) -> None:
        """Device-resident match writing to raw device addresses (e.g. rows of a peer-mapped image
        from shared_open): disparity rows at disp_ptr + r * disp_pitch, corrmap likewise."""
        p0, n, rows, cols, pitch, depth = self._stack_info(stack0)
        p1, n1, rows1, cols1, pitch1, depth1 = self._stack_info(stack1)
        if (n1, rows1, cols1, pitch1, depth1) != (n, rows, cols, pitch, depth):
            raise BicosError("stack0 and stack1 differ in length, size, type or pitch")
        ccfg = cfg.to_c()
        _check(lib().bicos_b200_match(self._h, p0, p1, n, rows, cols, pitch, depth, ctypes.byref(ccfg), disp_ptr,
                                      disp_pitch, corr_ptr, corr_pitch, self._stream()))

    def match_host(self, stack0, stack1, cfg: Config, out=None):
        """Host-resident match on numpy arrays / CPU tensors [n, rows, cols]; H2D and D2H included."""
        res = self.match_host_begin(stack0, stack1, cfg, out)
        self.match_host_end()
        return res

    def match_host_begin(self, stack0, stack1, cfg: Config, out=None):
        """Enqueue a host-resident match and return its (disparity, corrmap) buffers at once; they
        hold the result only after match_host_end(). One match in flight per handle: keep several
        frames in flight with several handles. The inputs must stay alive (and should be pinned)
        until match_host_end()."""
        import numpy as np

        def as_np(a):
            if hasattr(a, "numpy") and not isinstance(a, np.ndarray):
                a = a.numpy()
            return a

        s0, s1 = as_np(stack0), as_np(stack1)
        if s0.shape != s1.shape or s0.dtype != s1.dtype or s0.ndim != 3:
            raise BicosError("stack0 and stack1 differ")
        if s0.dtype == np.uint8:
            depth = DEPTH_8U
        elif s0.dtype == np.uint16:
            depth = DEPTH_16U
        else:
            raise BicosError("bad input depths, only uint8 and uint16 are supported")
        n, rows, cols = s0.shape
        # C-contiguous stacks are passed as views (the library then uploads whole bands with one
        # strided copy); anything else is made dense plane by plane
        planes0 = [s0[t] if s0[t].flags.c_contiguous else np.ascontiguousarray(s0[t]) for t in range(n)]
        planes1 = [s1[t] if s1[t].flags.c_contiguous else np.ascontiguousarray(s1[t]) for t in range(n)]
        ccfg = cfg.to_c()
        dt = lib().bicos_b200_disparity_type(ctypes.byref(ccfg))
        ct = lib().bicos_b200_corrmap_type(ctypes.byref(ccfg))
        if out is None:
            disp = np.empty((rows, cols), dtype=np.int16 if dt == TYPE_16S else np.float32)
            corr = np.empty((rows, cols), dtype=np.float64 if ct == TYPE_64F else np.float32) if ct else None
        else:
            try:
                out = tuple(as_np(o) if o is not None else None for o in out)
            except TypeError:
                raise BicosError("out must be a (disparity, corrmap) pair") from None
            disp, corr = self._check_out(ccfg, out, rows, cols)
        _check(lib().bicos_b200_match_host_begin(
            self._h, _ptr_array([p.ctypes.data for p in planes0]), _ptr_array([p.ctypes.data for p in planes1]),
            n, rows, cols, depth, ctypes.byref(ccfg), disp.ctypes.data,
            corr.ctypes.data if corr is not None else None))
        self._host_keepalive = (s0, s1, planes0, planes1, disp, corr)
        return disp, corr

    def match_host_end(self) -> None:
        _check(lib().bicos_b200_match_host_end(self._h))
        self._host_keepalive = None

    def set_overlap(self, enabled: bool) -> None:
        """False: every kernel of a match one after the other on the caller's stream (bicos_b200_set_overlap)."""
        _check(lib().bicos_b200_set_overlap(self._h, int(enabled)))

    def set_profiling(self, enabled: bool) -> None:
        """Record CUDA events around the three stages of every match (resets the accumulators)."""
        _check(lib().bicos_b200_set_profiling(self._h, int(enabled)))

    def stage_times(self):
        """(ms_transform, ms_search, ms_refine) accumulated since set_profiling(True), and the match count."""
        ms = (ctypes.c_double * 3)()
        cnt = ctypes.c_longlong()
        _check(lib().bicos_b200_stage_times(self._h, ms, ctypes.byref(cnt)))
        return [float(v) for v in ms], int(cnt.value)

    def synchronize(self) -> None:
        _check(lib().bicos_b200_synchronize(self._h, self._stream()))


class SharedImage:
    """A device image that other processes' GPUs can store into over NVLink (C ABI
    bicos_b200_shared_*): `SharedImage.create` on the assembling rank, `SharedImage.open(handle)`
    on the others. `tensor()` aliases the memory as a torch tensor (owner side)."""

    def __init__(self, device: int, ptr: int, rows: int, cols: int, dtype, owner: bool, handle: bytes = b""):
        self.device, self.ptr, self.rows, self.cols, self.dtype, self.owner, self.handle = \
            device, ptr, rows, cols, dtype, owner, handle

    @staticmethod
    def _itemsize(dtype) -> int:
        import torch

        return torch.empty((), dtype=dtype).element_size()

    @classmethod
    def create(cls, device: int, rows: int, cols: int, dtype) -> "SharedImage":
        ptr = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().bicos_b200_shared_alloc(device, rows * cols * cls._itemsize(dtype), ctypes.byref(ptr), handle))
        return cls(device, ptr.value, rows, cols, dtype, True, handle.raw)

    @classmethod
    def open(cls, device: int, handle: bytes, rows: int, cols: int, dtype) -> "SharedImage":
        ptr = ctypes.c_void_p()
        _check(lib().bicos_b200_shared_open(device, ctypes.create_string_buffer(handle, IPC_HANDLE_BYTES), ctypes.byref(ptr)))
        return cls(device, ptr.value, rows, cols, dtype, False)

    @property
    def pitch(self) -> int:
        return self.cols * self._itemsize(self.dtype)

    def row_ptr(self, row: int) -> int:
        return self.ptr + row * self.pitch

    def tensor(self):
        import torch

        typestr = {torch.float32: "<f4", torch.float64: "<f8", torch.int16: "<i2"}[self.dtype]

        class _Alias:
            __cuda_array_interface__ = {"shape": (self.rows, self.cols), "typestr": typestr,
                                        "data": (self.ptr, False), "version": 2}

        return torch.as_tensor(_Alias(), device=torch.device("cuda", self.device))

    def close(self) -> None:
        if self.ptr:
            fn = lib().bicos_b200_shared_free if self.owner else lib().bicos_b200_shared_close
            _check(fn(self.device, self.ptr))
            self.ptr = 0
