"""Per-pixel disparity windows (Handle.match_windows) against the range and the full row, on bench.py's workload.

2 x 33 uint8 2048 x 1536 stacks (LIMITED, thr 0.96, min_var 2.0, subpixel 0.1, Consistency{1}), matched one frame at a
time. Configurations:
  unranged            Handle.match, the whole row (the reference for the agreement column)
  range[14,77]        Handle.match with Config.disparity_range = (14, 77)
  windows[14,77]      constant window maps (14, 77): must equal the range bit for bit
  prior+-2, prior+-4  windows_from_disparity of synth's true disparity (17..75 px) with margin 2 / 4
  previous+-2         windows_from_disparity of the previous frame's unranged match, margin 2 (invalid pixels: the row)
  previous+-2/[14,77] the same, invalid pixels falling back to the range [14, 77]
  windows[14,77]/2    the constant windows with every other block of 128 columns empty (a region of interest)
For each it reports per match the search stage's device time (bicos_b200_stage_times), the whole match's time (CUDA
events around back-to-back matches), Mpx/s, the kernel that ran, and the share of pixels equal to the unranged result
(disparity and corrmap both). Configurations are measured in interleaved rounds in one process, medians over rounds.
The card's name and power limit are read in the same run.

    python tools/bench_windows.py [--rounds 5] [--steps 5] [--out FILE]
"""

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libbicos_b200 as lb  # noqa: E402
from libbicos_b200 import synth  # noqa: E402
from tools.bench_range import gpu_info  # noqa: E402

N_IMAGES, ROWS, COLS, FRAMES = 33, 1536, 2048, 4
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
RANGE = (14, 77)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5, help="passes over the frames per configuration and round")
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    h = lb.Handle(0)
    made = [synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=f, xp=torch, device="cuda") for f in range(FRAMES)]
    frames = [(l, r) for l, r, _ in made]
    truth = [torch.as_tensor(t, device="cuda", dtype=torch.float32) for _, _, t in made]
    cfg = lb.Config(**CFG)
    unranged = [h.match(l, r, cfg) for l, r in frames]

    def const(lo, hi):
        return (torch.full((ROWS, COLS), lo, dtype=torch.int16, device="cuda"),
                torch.full((ROWS, COLS), hi, dtype=torch.int16, device="cuda"))

    masked = const(*RANGE)
    blocks = (torch.arange(COLS, device="cuda") // 128) % 2 == 1
    masked[1][:, blocks] = RANGE[0] - 1  # min > max: empty
    windows = {
        "windows[14,77]": [const(*RANGE)] * FRAMES,
        "prior+-2": [h.windows_from_disparity(t, 2) for t in truth],
        "prior+-4": [h.windows_from_disparity(t, 4) for t in truth],
        "previous+-2": [h.windows_from_disparity(unranged[(f - 1) % FRAMES][0], 2) for f in range(FRAMES)],
        "previous+-2/[14,77]": [h.windows_from_disparity(unranged[(f - 1) % FRAMES][0], 2, RANGE) for f in range(FRAMES)],
        "windows[14,77]/2": [masked] * FRAMES,
    }
    names = ["unranged", "range[14,77]"] + list(windows)

    def run(name, f, out=None):
        l, r = frames[f]
        if name == "unranged":
            return h.match(l, r, cfg, out=out)
        if name == "range[14,77]":
            return h.match(l, r, lb.Config(disparity_range=RANGE, **CFG), out=out)
        return h.match_windows(l, r, windows[name][f], cfg, out=out)

    outs = {name: [run(name, f) for f in range(FRAMES)] for name in names}
    torch.cuda.synchronize()
    kernels, agree = {}, {}
    ref = [(d.cpu().numpy(), c.cpu().numpy()) for d, c in unranged]
    for name in names:
        run(name, 0, outs[name][0])
        kernels[name] = lb.last_search_kernel()
        got = [(d.cpu().numpy(), c.cpu().numpy()) for d, c in outs[name]]
        agree[name] = float(np.mean([np.mean(((g[0] == w[0]) | (np.isnan(g[0]) & np.isnan(w[0])))
                                             & ((g[1] == w[1]) | (np.isnan(g[1]) & np.isnan(w[1])))) for g, w in zip(got, ref)]))
    same_bits = all(np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)
                    for x, y in zip(outs["range[14,77]"], outs["windows[14,77]"]) for a, b in zip(x, y))

    search_ms = {name: [] for name in names}
    match_ms = {name: [] for name in names}
    for _ in range(args.rounds):
        for name in names:
            for f in range(FRAMES):  # warm-up
                run(name, f, outs[name][f])
            h.set_profiling(True)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(args.steps):
                for f in range(FRAMES):
                    run(name, f, outs[name][f])
            ev1.record()
            stages, count = h.stage_times()
            h.set_profiling(False)
            match_ms[name].append(ev0.elapsed_time(ev1) / (args.steps * FRAMES))
            search_ms[name].append(stages[1] / count)

    lines = []
    for name in names:
        s, m = float(np.median(search_ms[name])), float(np.median(match_ms[name]))
        lines.append(dict(config=name, search_ms=round(s, 4), match_ms=round(m, 4), mpx_per_s=round(ROWS * COLS / (m * 1e-3) / 1e6, 1),
                          kernel=kernels[name], same_as_unranged=round(agree[name], 5),
                          match_ms_spread=[round(min(match_ms[name]), 4), round(max(match_ms[name]), 4)]))
    lines.append(dict(constant_windows_equal_range_bitwise=same_bits, gpu=gpu_info(),
                      workload=f"2x{N_IMAGES} uint8 {COLS}x{ROWS}, {CFG}", rounds=args.rounds, matches_per_round=args.steps * FRAMES))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
