"""Generate tests/golden/remap/remap_cv2.npz: inputs and OpenCV's cv2.remap outputs for the rectification stage.

Needs cv2 (run once where it is installed): python tests/golden/make_remap_golden.py
tests/test_rectify.py compares its numpy restatement of the remap semantics (and, on the GPU, Handle.remap) with the
stored outputs, so that the comparison with OpenCV runs where cv2 is not installed. Stored: one uint8 and one uint16
source of 37 x 53 and, per case, the float32 maps [48, 67] and cv2.remap(src, map_x, map_y, INTER_LINEAR,
BORDER_CONSTANT, 0) of both sources:
  random   coordinates uniform over [-3, src + 2], reaching outside the image on every side
  ties     coordinates k / 64: every sixty-fourth is a rounding tie of the 1/32 quantisation
  special  NaN, +-inf, +-1e6, +-3e9, -0.5, -0.99, -1.02 and src - 1 +- 0.5 in either map, against ordinary values
"""
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_ROWS, SRC_COLS = 37, 53
ROWS, COLS = 48, 67


def cases(rng):
    yield "random", (rng.uniform(-3, SRC_COLS + 2, (ROWS, COLS)), rng.uniform(-3, SRC_ROWS + 2, (ROWS, COLS)))
    yield "ties", (rng.integers(-3 * 64, (SRC_COLS + 2) * 64, (ROWS, COLS)) / 64.0,
                   rng.integers(-3 * 64, (SRC_ROWS + 2) * 64, (ROWS, COLS)) / 64.0)
    special = np.array([np.nan, np.inf, -np.inf, 1e6, -1e6, 3e9, -3e9, -0.5, -0.99, -1.02])
    mx = rng.uniform(-1, SRC_COLS, (ROWS, COLS))
    my = rng.uniform(-1, SRC_ROWS, (ROWS, COLS))
    pick = rng.random((ROWS, COLS))
    mx = np.where(pick < 0.25, rng.choice(np.r_[special, SRC_COLS - 1.5, SRC_COLS - 0.5], (ROWS, COLS)), mx)
    my = np.where((pick > 0.2) & (pick < 0.45), rng.choice(np.r_[special, SRC_ROWS - 1.5, SRC_ROWS - 0.5], (ROWS, COLS)), my)
    yield "special", (mx, my)


def main():
    rng = np.random.default_rng(2026)
    out = dict(src8=rng.integers(0, 256, (SRC_ROWS, SRC_COLS), dtype=np.uint8),
               src16=rng.integers(0, 65536, (SRC_ROWS, SRC_COLS), dtype=np.uint16))
    out["src16"][:4] = 65535  # saturation at the top of the range
    for name, (mx, my) in cases(rng):
        mx, my = mx.astype(np.float32), my.astype(np.float32)
        out[f"{name}_mx"], out[f"{name}_my"] = mx, my
        for src in ("src8", "src16"):
            out[f"{name}_{src}"] = cv2.remap(out[src], mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    out["cv2_version"] = np.array(cv2.__version__)
    os.makedirs(os.path.join(HERE, "remap"), exist_ok=True)
    # a directory of its own: tests/golden/*.npz are the match fixtures of make_golden.py
    np.savez_compressed(os.path.join(HERE, "remap", "remap_cv2.npz"), **out)


if __name__ == "__main__":
    main()
