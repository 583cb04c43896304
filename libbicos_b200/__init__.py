"""libbicos_b200 -- a B200-native (sm_100a) implementation of libBICOS's matching hot path.

Layout:
  csrc/            hand-written CUDA kernels (transform, search, refine), the C ABI
                   (include/bicos_b200.h), BICOS::match (include/BICOS/match.hpp) and the
                   reference's Python FFI (include/pybicos_c.h)
  capi.py          ctypes binding of the C ABI for callers holding torch CUDA tensors
  pybicos/         drop-in for the reference's ``pybicos`` module
  sharding.py      row- / frame-sharding across GPUs with torch.distributed
  synth.py         seeded synthetic stereo stacks (tests and bench)

The product path is CUDA only. Importing this package does not load the shared library;
the first call does, and fails loudly if it has not been built.
"""

from .capi import (BicosError, Config, Handle, RectifyMaps, SharedImage, descriptor_words, last_search_kernel,  # noqa: F401
                   lib, search_engine, set_search_engine)

__all__ = ["BicosError", "Config", "Handle", "RectifyMaps", "SharedImage", "descriptor_words", "last_search_kernel", "lib",
           "search_engine", "set_search_engine"]
