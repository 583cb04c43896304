"""CPU tests of the boundary: both shared libraries load, export every symbol the headers
declare, the struct layouts match what the reference's Python module declares, and the product
path fails loudly (no fallback) when there is no CUDA device."""

import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__

    if not (os.path.exists(os.path.join(ROOT, "libbicos_b200", "libbicos_b200.so"))
            and os.path.exists(os.path.join(ROOT, "libbicos_b200", "pybicos", "pybicos_c.so"))):
        __graft_entry__.build()
    return True


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:bicos_b200|BICOS)_[A-Za-z0-9_]+)\s*\(", text)))


def test_c_abi_exports_every_declared_symbol(built):
    import libbicos_b200 as lb

    names = _declared("bicos_b200.h")
    assert len(names) >= 17 and set(lb.capi.EXPORTS) == set(names)
    L = ctypes.CDLL(lb.capi.LIB_PATH)
    for name in names:
        assert hasattr(L, name), name


def test_pybicos_c_exports_the_reference_ffi(built):
    names = _declared("pybicos_c.h")
    assert set(names) >= {"BICOS_CreateDefaultConfig", "BICOS_FreeConfig", "BICOS_FreeResult", "BICOS_Match",
                          "BICOS_InvalidDisparityFloat", "BICOS_InvalidDisparityInt16"}
    L = ctypes.CDLL(os.path.join(ROOT, "libbicos_b200", "pybicos", "pybicos_c.so"))
    for name in names:
        assert hasattr(L, name), name
    L.BICOS_InvalidDisparityFloat.restype = ctypes.c_float
    L.BICOS_InvalidDisparityInt16.restype = ctypes.c_int16
    assert np.isnan(L.BICOS_InvalidDisparityFloat()) and L.BICOS_InvalidDisparityInt16() == -32768


def test_config_defaults_and_layout(built):
    from libbicos_b200 import pybicos

    cfg = pybicos.Config()
    c = cfg._c_config.contents
    # reference src/pybicos_c.cpp:92-108
    assert (c.nxcorr_threshold, c.subpixel_step, c.min_variance) == (0.5, -1.0, -1.0)
    assert (c.mode, c.precision, c.variant_type, c.max_lr_diff, c.no_dupes) == (0, 0, 0, 1, 0)
    assert ctypes.sizeof(c) == 32  # 3 floats + 5 ints, as pybicos/__init__.py:41-51 declares
    cfg.set_consistency(3, True)
    cfg.subpixel_step = 0.25
    cfg.mode = pybicos.TransformMode.FULL
    cfg.precision = pybicos.Precision.DOUBLE
    assert cfg.variant == {"type": "Consistency", "max_lr_diff": 3, "no_dupes": True}
    assert cfg.subpixel_step == 0.25 and cfg.min_variance is None
    assert cfg.mode is pybicos.TransformMode.FULL and cfg.precision is pybicos.Precision.DOUBLE
    cfg.set_no_duplicates()
    assert cfg.variant == "NoDuplicates"
    assert np.isnan(pybicos.invalid_disparity(np.float32)) and pybicos.invalid_disparity(np.int16) == -32768


def test_capi_config_mapping(built):
    import libbicos_b200 as lb

    c = lb.Config(nxcorr_threshold=None, subpixel_step=0.1, consistency=True, max_lr_diff=2, no_dupes=True).to_c()
    assert c.nxcorr_threshold == -1.0 and abs(c.subpixel_step - 0.1) < 1e-7 and c.min_variance == -1.0
    assert (c.variant_type, c.max_lr_diff, c.no_dupes) == (1, 2, 1)
    assert lb.Config().flags == 1 and lb.Config(consistency=True).flags == 2
    assert lb.Config(consistency=True, no_dupes=True).flags == 3
    # descriptor width choice of the reference dispatch (src/impl/cpu.cpp:122-156)
    assert [lb.descriptor_words(n) for n in (2, 9, 10, 17, 18, 33, 34, 65)] == [1, 1, 2, 2, 4, 4, 8, 8]
    assert [lb.descriptor_words(n, True) for n in (2, 6, 7, 8, 9, 12, 13, 16)] == [1, 1, 2, 2, 4, 4, 8, 8]
    with pytest.raises(lb.BicosError, match="would require 257 bits"):
        lb.descriptor_words(66)
    with pytest.raises(lb.BicosError, match="363 bits"):
        lb.descriptor_words(20, True)


def test_no_fallback_without_gpu(built):
    import torch

    if torch.cuda.is_available():
        pytest.skip("this test is about machines without a GPU")
    import libbicos_b200 as lb
    from libbicos_b200 import pybicos

    with pytest.raises(lb.BicosError):
        lb.Handle(0)
    img = [np.zeros((8, 8), np.uint8)] * 3
    with pytest.raises(RuntimeError, match="BICOS matching failed"):
        pybicos.match(img, img)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under libbicos_b200/ may reference it."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "libbicos_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in text and "from oracle" not in text and "bicos_oracle" not in text, f
    out = subprocess.run([sys.executable, "-c",
                          "import sys; sys.path.insert(0, %r); import libbicos_b200, libbicos_b200.sharding; "
                          "print('oracle' in sys.modules)" % ROOT], capture_output=True, text=True)
    assert out.stdout.strip() == "False"


def test_reference_pybicos_module_loads_our_library(built, tmp_path):
    """The UNMODIFIED reference pybicos/__init__.py binds our pybicos_c.so (drop-in at the FFI)."""
    import oracle

    ref_init = os.path.join(oracle.REFERENCE_DIR, "pybicos", "__init__.py")
    if not oracle.REFERENCE_DIR or not os.path.exists(ref_init):
        pytest.skip("needs a checkout of the reference project (BICOS_REFERENCE_DIR)")
    pkg = tmp_path / "pybicos"
    pkg.mkdir()
    os.symlink(ref_init, pkg / "__init__.py")
    os.symlink(os.path.join(ROOT, "libbicos_b200", "pybicos", "pybicos_c.so"), pkg / "pybicos_c.so")
    code = ("import sys; sys.path.insert(0, %r); import pybicos; c = pybicos.Config(); c.set_consistency(2, True); "
            "c.precision = pybicos.Precision.DOUBLE; print(c.nxcorr_threshold, c.variant, c.precision.name)" % str(tmp_path))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip() == "0.5 {'type': 'Consistency', 'max_lr_diff': 2, 'no_dupes': True} DOUBLE"


def test_reference_signature_with_opencv_types():
    """-DBICOS_WITH_OPENCV: BICOS::match takes cv::cuda::GpuMat images and a cv::cuda::Stream& as the reference does
    (include/match.hpp:31-41). Compile-only, against the stand-in headers of oracle/shim."""
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-DBICOS_WITH_OPENCV", "-I" + os.path.join(ROOT, "oracle", "shim"),
           "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
           os.path.join(ROOT, "tests", "cpp", "opencv_signature_check.cpp")]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


def test_host_out_buffers_are_validated_before_any_device_work(built):
    """Handle.match_host(out=...) refuses buffers of the wrong dtype / shape / layout before the C ABI is called
    (so this runs without a GPU: the check needs only the pure type queries of the library)."""
    import libbicos_b200 as lb

    h = lb.Handle.__new__(lb.Handle)  # no device needed for the validation path
    h._h = None
    left = np.zeros((3, 8, 16), np.uint8)
    cfg = lb.Config(nxcorr_threshold=0.5)
    good = np.empty((8, 16), np.float32)
    for out in ((np.empty((8, 16), np.int16), good), (good, None), (good, np.empty((8, 16), np.float64)),
                (np.empty((16, 8), np.float32).T, good), (np.empty((4, 16), np.float32), good), good):
        with pytest.raises(lb.BicosError, match="out "):
            h.match_host_begin(left, left, cfg, out=out)
    with pytest.raises(lb.BicosError, match="out corrmap must be None"):
        h.match_host_begin(left, left, lb.Config(nxcorr_threshold=None), out=(np.empty((8, 16), np.int16), good))


def test_last_search_kernel_starts_empty(built):
    import libbicos_b200 as lb

    assert isinstance(lb.last_search_kernel(), str)
