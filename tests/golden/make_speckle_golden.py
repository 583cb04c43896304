"""Generate tests/golden/speckles/speckles_cv2.npz: int16 disparities and OpenCV's cv2.filterSpeckles outputs.

Needs cv2 (run once where it is installed): python tests/golden/make_speckle_golden.py
tests/test_speckles.py compares its connected-components restatement of bicos_b200_filter_speckles (and, on the GPU,
Handle.filter_speckles) with the stored outputs, so that the comparison with OpenCV runs where cv2 is not installed.
Stored per case: `<name>_in` (int16 [rows, cols]), `<name>_out` = cv2.filterSpeckles(in, new_value, max_speckle_size,
max_diff) and `<name>_prm` = (new_value, max_speckle_size, max_diff) as float64. Every case either has new_value =
-32768 or no -32768 pixels, where the library's semantics and OpenCV's coincide:
  random_*      low-entropy random scenes (blobs of every size), with and without -32768 markers
  exact_size    bars of exactly max_speckle_size and max_speckle_size + 1 pixels
  diff0, diffneg, size0, sizeneg, sizeall    max_diff of 0 and -1, max_speckle_size of 0, -3 and rows * cols
  extremes_*    +-32767, +-1 and 0 neighbours with max_diff 32767 and 32766 (OpenCV's IPP path truncates a max_diff
                beyond 32767 to int16, so larger ones are checked against the scan-order port instead)
  ties_*        new_value and max_diff halfway between two integers (cvRound rounds half to even)
"""
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MARKER = -32768


def _random(rng, rows, cols, levels, markers):
    d = rng.integers(0, levels, (rows, cols)).astype(np.int16)
    if markers:
        d[rng.random((rows, cols)) < 0.06] = MARKER
    return d


def _bars(rows, cols, k):
    """Background of neighbours 1000 apart; horizontal bars of k (value 7) and k + 1 (value 9) pixels."""
    r, c = np.mgrid[0:rows, 0:cols]
    d = np.where((r + c) % 2 == 0, 1000, 3000).astype(np.int16)
    for y in range(1, rows - 1, 3):
        x = 1
        while x + 2 * k + 4 < cols:
            d[y, x:x + k] = 7
            d[y, x + k + 2:x + 2 * k + 3] = 9
            x += 2 * k + 5
    return d


def cases(rng):
    yield "random_marker", _random(rng, 61, 93, 4, True), (MARKER, 5, 0)
    yield "random_d1", _random(rng, 64, 130, 7, False), (0, 12, 1)
    yield "random_big", _random(rng, 150, 260, 3, True), (MARKER, 40, 0)
    yield "exact_size", _bars(30, 80, 6), (MARKER, 6, 0)
    yield "diff0", _random(rng, 40, 50, 3, False), (-1, 8, 0)
    yield "diffneg", _random(rng, 40, 50, 3, True), (MARKER, 8, -1)
    yield "size0", _random(rng, 20, 30, 2, True), (MARKER, 0, 0)
    yield "sizeneg", _random(rng, 20, 30, 2, True), (MARKER, -3, 0)
    yield "sizeall", _random(rng, 20, 30, 5, True), (MARKER, 600, 1)
    ext = rng.choice(np.array([32767, -32767, 0, 1, -1], np.int16), (33, 47))
    yield "extremes_32767", ext, (MARKER, 6, 32767)
    yield "extremes_32766", ext, (MARKER, 6, 32766)
    yield "ties_low", _random(rng, 40, 60, 6, False), (2.5, 5, 1.5)  # new 2, diff 2
    yield "ties_high", _random(rng, 40, 60, 6, False), (3.5, 5, 0.5)  # new 4, diff 0
    yield "ties_neg", _random(rng, 40, 60, 6, True), (-32768.5, 5, 2.5)  # new -32768, diff 2


def main():
    rng = np.random.default_rng(7)
    out = {}
    for name, d, (new_value, size, diff) in cases(rng):
        got, _ = cv2.filterSpeckles(d.copy(), new_value, size, diff)
        out[name + "_in"] = d
        out[name + "_out"] = got
        out[name + "_prm"] = np.array([new_value, size, diff], dtype=np.float64)
    os.makedirs(os.path.join(HERE, "speckles"), exist_ok=True)
    np.savez_compressed(os.path.join(HERE, "speckles", "speckles_cv2.npz"), **out)


if __name__ == "__main__":
    main()
