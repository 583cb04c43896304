"""Disparity-range search against the full-row search, on bench.py's workload.

2 x 33 uint8 2048 x 1536 stacks (LIMITED, thr 0.96, min_var 2.0, subpixel 0.1, Consistency{1}), matched one frame at a
time with Handle.match. For the unranged configuration and for windows of D + 1 = 64, 128, 256, 512 disparities
(centred on 46 px, so that every true disparity of the synthetic scene, 17..75 px, is inside), it reports per match:
the search stage's device time (bicos_b200_stage_times), the whole match's time (CUDA events around back-to-back
matches), Mpx/s, the kernel that ran, and the share of pixels whose result equals the unranged one. Configurations are
measured in interleaved rounds in one process, medians over rounds. The crossover is the window width beyond which a
ranged match is slower than the unranged one (linear between the measured widths).

    python tools/bench_range.py [--rounds 5] [--steps 5] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libbicos_b200 as lb  # noqa: E402
from libbicos_b200 import synth  # noqa: E402

N_IMAGES, ROWS, COLS, FRAMES = 33, 1536, 2048, 4
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
WIDTHS = (64, 128, 256, 512)
CENTRE = 46


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return f"{name} ({q})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5, help="passes over the frames per configuration and round")
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    h = lb.Handle(0)
    frames = [synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=f, xp=torch, device="cuda")[:2] for f in range(FRAMES)]
    configs = [("unranged", None)] + [(f"D+1={w}", (CENTRE - w // 2, CENTRE - w // 2 + w - 1)) for w in WIDTHS]
    outs = {name: [h.match(l, r, lb.Config(disparity_range=rng, **CFG)) for l, r in frames] for name, rng in configs}
    torch.cuda.synchronize()
    kernels, agree = {}, {}
    ref = [(d.cpu().numpy(), c.cpu().numpy()) for d, c in outs["unranged"]]
    for name, rng in configs:
        h.match(*frames[0], lb.Config(disparity_range=rng, **CFG), out=outs[name][0])
        kernels[name] = lb.last_search_kernel()
        got = [(d.cpu().numpy(), c.cpu().numpy()) for d, c in outs[name]]
        agree[name] = float(np.mean([np.mean((g[0] == w[0]) | (np.isnan(g[0]) & np.isnan(w[0]))) for g, w in zip(got, ref)]))

    search_ms = {name: [] for name, _ in configs}
    match_ms = {name: [] for name, _ in configs}
    for _ in range(args.rounds):
        for name, rng in configs:
            cfg = lb.Config(disparity_range=rng, **CFG)
            for (l, r), out in zip(frames, outs[name]):  # warm-up
                h.match(l, r, cfg, out=out)
            h.set_profiling(True)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(args.steps):
                for (l, r), out in zip(frames, outs[name]):
                    h.match(l, r, cfg, out=out)
            ev1.record()
            stages, count = h.stage_times()
            h.set_profiling(False)
            match_ms[name].append(ev0.elapsed_time(ev1) / (args.steps * FRAMES))
            search_ms[name].append(stages[1] / count)

    gpu = gpu_info()
    lines = []
    med = {name: (float(np.median(search_ms[name])), float(np.median(match_ms[name]))) for name, _ in configs}
    for name, rng in configs:
        s, m = med[name]
        lines.append(dict(config=name, disparity_range=rng, search_ms=round(s, 4), match_ms=round(m, 4),
                          mpx_per_s=round(ROWS * COLS / (m * 1e-3) / 1e6, 1), kernel=kernels[name],
                          same_as_unranged=round(agree[name], 5),
                          match_ms_spread=[round(min(match_ms[name]), 4), round(max(match_ms[name]), 4)]))
    full = med["unranged"][1]
    cross = None
    prev_w, prev_m = None, None
    for w in WIDTHS:
        m = med[f"D+1={w}"][1]
        if m > full:
            cross = w if prev_w is None else prev_w + (w - prev_w) * (full - prev_m) / (m - prev_m)
            break
        prev_w, prev_m = w, m
    lines.append(dict(crossover_window=round(cross, 1) if cross is not None else None,
                      note=("ranged match slower than unranged beyond this window width D + 1" if cross is not None
                            else f"every measured window (up to D + 1 = {WIDTHS[-1]}) is faster than the unranged match"),
                      gpu=gpu, workload=f"2x{N_IMAGES} uint8 {COLS}x{ROWS}, {CFG}", rounds=args.rounds,
                      matches_per_round=args.steps * FRAMES))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
