"""What the comparisons with the reference libBICOS build check against, stored so that they also run without it.

Tests that compare with the reference build (oracle.ref, oracle.refcuda) keep that live comparison when the build is
present. Without it they compare against the outputs written here:

* reference/outputs.json: a SHA-256 digest of every array those tests require to be identical (descriptors, disparity,
  corrmap), with a CRC of every input, so that a changed synthetic generator and a changed output fail differently;
* reference/outputs.npz: the arrays themselves where a test needs values: the tie-breaking search results and the
  double-precision disparity / corrmap (a seeded sample of pixels) of the reference CUDA build comparison.

The inputs below are those of the tests (keys name the test and its parameters).

    python tests/golden/make_reference_outputs.py [--source ref|port]

`--source ref` (the default) computes every output with the reference build (BICOS_REFERENCE_DIR, see oracle/);
the double-precision part needs a GPU for oracle.refcuda. `--source port` computes them with oracle.port, the C
restatement: on these inputs its outputs are the reference's, as long as bicos_oracle.c is unchanged since every one
of these comparisons passed against the reference build, which is how the committed files were made (see the
"source" field of the JSON file).
"""

import argparse
import hashlib
import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
JSON_PATH = os.path.join(HERE, "reference", "outputs.json")
NPZ_PATH = os.path.join(HERE, "reference", "outputs.npz")

# tests/test_oracle.py::test_port_matches_reference_build
BUILD_CASES = [(2, np.uint8, False), (3, np.uint16, True), (9, np.uint8, False), (12, np.uint8, True),
               (16, np.uint16, True), (20, np.uint16, False), (33, np.uint8, False), (65, np.uint8, False)]
BUILD_KWS = [dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.9, min_variance=2.0),
             dict(nxcorr_threshold=0.8, subpixel_step=0.1, consistency=True, max_lr_diff=1),
             dict(nxcorr_threshold=0.8, subpixel_step=0.3, consistency=True, max_lr_diff=0, no_dupes=True, min_variance=0.5)]
# tests/test_oracle.py::test_wide_extension_matches_reference_stage_templates
WIDE_CASES = [(17, np.uint8), (20, np.uint16), (21, np.uint16), (23, np.uint8)]
WIDE_KWS = [dict(nxcorr_threshold=None), dict(nxcorr_threshold=0.9, min_variance=2.0),
            dict(nxcorr_threshold=0.8, subpixel_step=0.25, consistency=True, max_lr_diff=1, no_dupes=True)]
# tests/test_gpu_parity.py::test_match_against_unmodified_reference
GPU_KWS = [dict(nxcorr_threshold=0.96, min_variance=2.0),
           dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)]
# tests/test_gpu_parity.py::test_double_precision_against_reference_cuda_build
DOUBLE_CASES = [(33, np.uint8, dict(nxcorr_threshold=0.9, min_variance=2.0, double=True)),
                (16, np.uint16, dict(nxcorr_threshold=0.9, mode_full=True, double=True, consistency=True))]
DOUBLE_SAMPLE = 4096  # corrmap pixels stored per case


def build_inputs(n, dtype, rows=40):
    from libbicos_b200 import synth

    return synth.make_stacks(n, 512, 150, dtype, seed=n, row0=130, rows=rows)[:2]


def gpu_inputs():
    from libbicos_b200 import synth

    return synth.make_stacks(33, 512, 400, np.uint8, seed=99, row0=256, rows=64)[:2]


def double_inputs(n, dtype):
    from libbicos_b200 import synth

    return synth.make_stacks(n, 512, 384, dtype, seed=41, row0=200, rows=64)[:2]


def tie_descriptors():
    """{k: (d0, d1)}: random low-entropy descriptors, drawn in the test's order."""
    rng = np.random.default_rng(0)
    out = {}
    for k in (1, 2, 4, 8, 12, 16):
        d0 = rng.integers(0, 8, size=(5, 90, k)).astype(np.uint32)
        d1 = rng.integers(0, 8, size=(5, 90, k)).astype(np.uint32)
        out[k] = (d0, d1)
    return out


def double_sample(rows, cols):
    return np.random.default_rng(41).choice(rows * cols, DOUBLE_SAMPLE, replace=False)


def digest(a):
    """SHA-256 of dtype, shape and values, equal exactly when np.array_equal(..., equal_nan=True) holds for arrays
    of one dtype and shape: every NaN becomes the one NaN and -0 becomes +0 first. None digests to None."""
    if a is None:
        return None
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), a.dtype.type(np.nan), a + a.dtype.type(0))
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def crc(*arrays):
    c = 0
    for a in arrays:
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return c


_stored = None


def stored():
    """(digests, arrays) as committed."""
    global _stored
    if _stored is None:
        with open(JSON_PATH) as f:
            digests = json.load(f)["digests"]
        _stored = digests, dict(np.load(NPZ_PATH))
    return _stored


def check_inputs(key, *arrays):
    assert stored()[0][f"{key}/inputs"] == crc(*arrays), f"{key}: inputs changed (synthetic generator): regenerate"


def check(key, a):
    """a must be identical to the reference's output stored under key."""
    assert digest(a) == stored()[0][key], f"{key}: differs from the reference's output"


def generate(source):
    import oracle

    if source == "ref":
        oracle.build(ref=True)
        assert oracle.ref.available(), "the reference build is missing: set BICOS_REFERENCE_DIR (see oracle/)"
        cpu, cuda = oracle.ref, oracle.refcuda
    else:
        oracle.build(ref=False)
        cpu, cuda = oracle.port, None
    digests, arrays = {}, {}

    for n, dtype, full in BUILD_CASES:
        key = f"port_build/{n}_{np.dtype(dtype).name}_{int(full)}"
        left, right = build_inputs(n, dtype)
        digests[f"{key}/inputs"] = crc(left, right)
        digests[f"{key}/desc"] = digest(cpu.descriptors(left, full))
        for i, kw in enumerate(BUILD_KWS):
            d, c = cpu.match(left, right, mode_full=full, **kw)
            digests[f"{key}/{i}/disp"], digests[f"{key}/{i}/corr"] = digest(d), digest(c)

    for n, dtype in WIDE_CASES:
        key = f"wide/{n}_{np.dtype(dtype).name}"
        left, right = build_inputs(n, dtype, rows=16)
        digests[f"{key}/inputs"] = crc(left, right)
        digests[f"{key}/desc"] = digest(cpu.descriptors(left, True, wide=True))
        for i, kw in enumerate(WIDE_KWS):
            d, c = cpu.match(left, right, mode_full=True, wide_descriptors=True, **kw)
            digests[f"{key}/{i}/disp"], digests[f"{key}/{i}/corr"] = digest(d), digest(c)

    for k, (d0, d1) in tie_descriptors().items():
        for flags in (1, 2, 3):
            arrays[f"ties_k{k}_f{flags}"] = cpu.bicos(d0, d1, flags, 2)

    left, right = gpu_inputs()
    digests["gpu_match/inputs"] = crc(left, right)
    for i, kw in enumerate(GPU_KWS):
        d, c = cpu.match(left, right, **kw)
        digests[f"gpu_match/{i}/disp"], digests[f"gpu_match/{i}/corr"] = digest(d), digest(c)

    for n, dtype, kw in DOUBLE_CASES:
        key = f"double_{n}"
        left, right = double_inputs(n, dtype)
        digests[f"{key}/inputs"] = crc(left, right)
        if cuda is not None:
            d, c = cuda.match(left, right, **kw)  # int16 disparity; corrmap cells never evaluated are uninitialised
        else:
            d, c = cpu.match(left, right, **kw)  # float32 disparity holding integers, NaN where never evaluated
            d = d.astype(np.int16)
        arrays[f"{key}_disp"] = d
        arrays[f"{key}_corr_sample"] = c.reshape(-1)[double_sample(*d.shape)]

    os.makedirs(os.path.dirname(JSON_PATH), exist_ok=True)
    with open(JSON_PATH, "w") as f:
        json.dump({"source": {"ref": "reference build (oracle.ref, oracle.refcuda)",
                              "port": "oracle.port (bicos_oracle.c), identical to the reference build on these inputs"}[source],
                   "digests": digests}, f, indent=0, sort_keys=True)
        f.write("\n")
    np.savez_compressed(NPZ_PATH, **arrays)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["ref", "port"], default="ref")
    generate(ap.parse_args().source)
